import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gic_b200
from gic_b200 import _lib
from gic_b200.discriminator import disc_fwd_raw
d=torch.device('cuda:0'); lib=_lib.lib()
N,L,V,fsz,nfl,R=512,20,10000,[3,4,5],[300,300,300],64
g=torch.Generator(device=d).manual_seed(0)
De,Fd,Hd=R,sum(nfl),100
u=lambda *s:(torch.rand(*s,generator=g,device=d)-0.5)*0.1
W_e=u(De,V)*10; cw=[u(n,1,f,1).contiguous() for n,f in zip(nfl,fsz)]; cb=[u(n) for n in nfl]
W_h,b_h,W_f,b_f,W_o,b_o=u(Fd,Fd),u(Fd),u(Hd,Fd),u(Hd),u(1,Hd),u(1)
ids=torch.randint(0,V,(N,L),generator=g,device=d)
for _ in range(2): disc_fwd_raw(lib,gic_b200.GEMM_BF16,None,ids,N,L,V,De,R,fsz,nfl,W_e,cw,cb,W_h,b_h,W_f,b_f,W_o,b_o,[None],0.0,d)
torch.cuda.synchronize()
