import os, sys, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
import gic_b200
from gic_b200 import _lib
from gic_b200.discriminator import disc_fwd_raw
d=torch.device('cuda:0'); lib=_lib.lib()
def run(N,L,V=10000,fsz=[3,4,5],nfl=[300,300,300],R=64):
    g=torch.Generator(device=d).manual_seed(0)
    De,Fd,Hd=R,sum(nfl),100
    u=lambda *s:(torch.rand(*s,generator=g,device=d)-0.5)*0.1
    W_e=u(De,V)*10; cw=[u(n,1,f,1).contiguous() for n,f in zip(nfl,fsz)]; cb=[u(n) for n in nfl]
    W_h,b_h,W_f,b_f,W_o,b_o=u(Fd,Fd),u(Fd),u(Hd,Fd),u(Hd),u(1,Hd),u(1)
    ids=torch.randint(0,V,(N,L),generator=g,device=d)
    gic_b200.prof_enable(True) if hasattr(gic_b200,'prof_enable') else None
    for flag,sl in (("0",""),("1",""),("1","2"),("1","3"),("1","6"),("1","8")):
        from gic_b200 import _lib
        _lib.set_option("GIC_CONV_MMA", int(flag))
        if sl: _lib.set_option("GIC_CONV_MMA_SLICES", int(sl))
        else: _lib.clear_option("GIC_CONV_MMA_SLICES")
        for _ in range(3): disc_fwd_raw(lib,gic_b200.GEMM_BF16,None,ids,N,L,V,De,R,fsz,nfl,W_e,cw,cb,W_h,b_h,W_f,b_f,W_o,b_o,[None],0.0,d)
        torch.cuda.synchronize()
        e0=torch.cuda.Event(enable_timing=True); e1=torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10): disc_fwd_raw(lib,gic_b200.GEMM_BF16,None,ids,N,L,V,De,R,fsz,nfl,W_e,cw,cb,W_h,b_h,W_f,b_f,W_o,b_o,[None],0.0,d)
        e1.record(); torch.cuda.synchronize()
        print(f"N={N} L={L} mma={flag} slices={sl or 'auto'}: disc fwd {e0.elapsed_time(e1)/10*1000:.1f} us")
run(256,20); run(512,20); run(4096,32)
