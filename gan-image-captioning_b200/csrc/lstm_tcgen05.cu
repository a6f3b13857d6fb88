// Fused LSTM decode step on the tensor cores (sm_100a): one kernel computes
//     gates = x W_ih^T + h W_hh^T + b_ih + b_hh            (both contractions accumulate into one TMEM tile)
//     i,f,g,o -> c' = sig(f) c + sig(i) tanh(g),  h' = sig(o) tanh(c')
// for one layer and one time step (src/generator.py:61).  It replaces two GEMM launches, the [B,4H] gates round
// trip through HBM and the cell kernel of the unfused path.
//
// Tiling: a CTA owns 128 batch rows x U hidden units (U = 8, 16 or 32, chosen so that the grid covers the SMs: at
// B = 256, H = 512 that is 2 x 64 CTAs of U = 8).  Its B operand tile is gate-interleaved: four U-row slabs of the
// weight matrix (rows g*H + j0 .. j0+U-1 for g = i,f,g,o) are TMA-loaded next to each other, so the 4U accumulator
// columns are [i(U) | f(U) | g(U) | o(U)] of the same U units and the cell update is an epilogue on the TMEM tile.  The k loop runs over ceil(In/32) blocks of (x, W_ih) followed by ceil(H/32) blocks of
// (h, W_hh).  Warp roles as in gemm_tcgen05.cu.
#include "tcgen05_common.cuh"

namespace gic {
namespace tc {

template <int U>
struct LstmCfg {
  static constexpr int A_BYTES = BM * BK * 4;            // 16 KB
  static constexpr int B_BYTES = 4 * U * BK * 4;         // 4 gates x U rows x 128 B
  static constexpr int STAGE = A_BYTES + B_BYTES;
  static constexpr int STAGES = (U == 32) ? 6 : 8;
  static constexpr int SMEM = STAGES * STAGE + 1024 + 256;
  static constexpr uint32_t TMEM_COLS = (4 * U < 32) ? 32 : 4 * U;
};

template <int U>
__global__ void __launch_bounds__(NTHREADS, 1)
lstm_step_tf32_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmH,
                      const __grid_constant__ CUtensorMap tmWih, const __grid_constant__ CUtensorMap tmWhh, int B,
                      int H, int In, const float* __restrict__ b_ih, const float* __restrict__ b_hh,
                      const float* __restrict__ c_prev, float* __restrict__ acts, float* __restrict__ c_out,
                      float* __restrict__ h_out, float* __restrict__ htop, int L, int t) {
  using S = LstmCfg<U>;
  constexpr int LSTM_STAGES = S::STAGES, LSTM_STAGE = S::STAGE;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + LSTM_STAGES * LSTM_STAGE);
  uint64_t* empty = full + LSTM_STAGES;
  uint64_t* tmem_full = empty + LSTM_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int j0 = blockIdx.x * U, m0 = blockIdx.y * BM;
  const int nkb1 = (In + BK - 1) / BK, nkb2 = (H + BK - 1) / BK, nkb = nkb1 + nkb2;
  constexpr uint32_t TMEM_COLS = S::TMEM_COLS;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmX) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmWih) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmH) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmWhh) : "memory");
    for (int s = 0; s < LSTM_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(tmem_full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();                      // everything above overlapped the previous kernel of the decode chain
  pdl_trigger();

  if (warp == 0) {
    if (lane == 0) {
      for (int kb = 0; kb < nkb; ++kb) {
        const int s = kb % LSTM_STAGES;
        const uint32_t ph = (kb / LSTM_STAGES) & 1;
        mbar_wait(&empty[s], ph ^ 1);
        uint8_t* sa = smem + s * LSTM_STAGE;
        uint8_t* sb = sa + BM * BK * 4;
        mbar_expect_tx(&full[s], LSTM_STAGE);
        const bool first = kb < nkb1;
        const int k0 = (first ? kb : kb - nkb1) * BK;
        tma_load_2d(sa, first ? &tmX : &tmH, &full[s], k0, m0);
#pragma unroll
        for (int g = 0; g < 4; ++g) tma_load_2d(sb + g * (U * 128), first ? &tmWih : &tmWhh, &full[s], k0, g * H + j0);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc(0, 0, 4 * U);
      for (int kb = 0; kb < nkb; ++kb) {
        const int s = kb % LSTM_STAGES;
        const uint32_t ph = (kb / LSTM_STAGES) & 1;
        mbar_wait(&full[s], ph);
        tcgen05_fence_after();
        const uint32_t sa = smem_u32(smem + s * LSTM_STAGE);
        const uint32_t sb = sa + BM * BK * 4;
#pragma unroll
        for (int k = 0; k < BK / UMMA_K; ++k)
          umma_tf32(tmem_base, make_desc(sa + k * 32, 16, 1024, 2), make_desc(sb + k * 32, 16, 1024, 2), idesc,
                    (kb > 0 || k > 0) ? 1u : 0u);
        umma_commit(&empty[s]);
      }
      umma_commit(tmem_full);
    }
  } else {
    // ===== epilogue: LSTM cell on the accumulator tile =====
    const int q = warp & 3;
    const int b = m0 + q * 32 + lane;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
    // the first unit group's previous cell state and biases are fetched while the main loop runs
    float cp0[8], bs0[4][8];
    {
      const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
      const bool ok = b < B;
      *reinterpret_cast<float4*>(cp0) = ok ? *reinterpret_cast<const float4*>(c_prev + (size_t)b * H + j0) : z4;
      *reinterpret_cast<float4*>(cp0 + 4) = ok ? *reinterpret_cast<const float4*>(c_prev + (size_t)b * H + j0 + 4) : z4;
#pragma unroll
      for (int g = 0; g < 4; ++g) {
#pragma unroll
        for (int h4 = 0; h4 < 2; ++h4) {
          const float4 x = __ldg(reinterpret_cast<const float4*>(b_ih + g * H + j0) + h4);
          const float4 y = __ldg(reinterpret_cast<const float4*>(b_hh + g * H + j0) + h4);
          bs0[g][4 * h4 + 0] = x.x + y.x; bs0[g][4 * h4 + 1] = x.y + y.y;
          bs0[g][4 * h4 + 2] = x.z + y.z; bs0[g][4 * h4 + 3] = x.w + y.w;
        }
      }
    }
    mbar_wait(tmem_full, 0);
    tcgen05_fence_after();
#pragma unroll 1
    for (int u0 = 0; u0 < U; u0 += 8) {
      uint32_t ri[8], rf[8], rg[8], ro[8];
      tmem_ld8(lane_addr + 0 * U + u0, ri);
      tmem_ld8(lane_addr + 1 * U + u0, rf);
      tmem_ld8(lane_addr + 2 * U + u0, rg);
      tmem_ld8(lane_addr + 3 * U + u0, ro);
      if (b < B) {
        const int j = j0 + u0;
        float cp[8], bs[4][8], ai[8], af[8], ag[8], ao[8], cn[8], hn[8];
        if (u0 == 0) {
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            cp[e] = cp0[e];
            bs[0][e] = bs0[0][e]; bs[1][e] = bs0[1][e]; bs[2][e] = bs0[2][e]; bs[3][e] = bs0[3][e];
          }
        } else {
          *reinterpret_cast<float4*>(cp) = *reinterpret_cast<const float4*>(c_prev + (size_t)b * H + j);
          *reinterpret_cast<float4*>(cp + 4) = *reinterpret_cast<const float4*>(c_prev + (size_t)b * H + j + 4);
#pragma unroll
          for (int g = 0; g < 4; ++g)
#pragma unroll
            for (int e = 0; e < 8; ++e) bs[g][e] = b_ih[g * H + j + e] + b_hh[g * H + j + e];
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float pi = __uint_as_float(ri[e]) + bs[0][e];
          const float pf = __uint_as_float(rf[e]) + bs[1][e];
          const float pg = __uint_as_float(rg[e]) + bs[2][e];
          const float po = __uint_as_float(ro[e]) + bs[3][e];
          ai[e] = sigmoidf_acc(pi); af[e] = sigmoidf_acc(pf); ag[e] = tanhf(pg); ao[e] = sigmoidf_acc(po);
          cn[e] = af[e] * cp[e] + ai[e] * ag[e];
          hn[e] = ao[e] * tanhf(cn[e]);
        }
        auto st8 = [](float* dst, const float* v) {
          *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
          *reinterpret_cast<float4*>(dst + 4) = make_float4(v[4], v[5], v[6], v[7]);
        };
        if (acts) {                  // saved for the backward pass; rollouts (no backward) pass nullptr
          float* arow = acts + (size_t)b * 4 * H + j;
          st8(arow, ai); st8(arow + H, af); st8(arow + 2 * H, ag); st8(arow + 3 * H, ao);
        }
        st8(c_out + (size_t)b * H + j, cn);
        st8(h_out + (size_t)b * H + j, hn);
        if (htop) st8(htop + ((size_t)b * L + t) * H + j, hn);
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS));
  }
}

}  // namespace tc

// One LSTM layer / time step on the tensor cores.  handled = false (nothing launched) when the shape does not fit
// the kernel (H % 32, TMA alignment); the caller then runs the unfused GEMM + cell path.
int lstm_step_tc(const float* x, int In, const float* h_prev, const float* W_ih, const float* W_hh, const float* b_ih,
                 const float* b_hh, const float* c_prev, int B, int H, float* acts, float* c_out, float* h_out,
                 float* htop, int L, int t, cudaStream_t stream, bool* handled) {
  using namespace tc;
  *handled = false;
  if (B <= 0 || (H % 8) || (In % 4) || In < 4) return GIC_OK;
  const void* ptrs[] = {x, h_prev, W_ih, W_hh, c_prev, acts ? acts : h_out, c_out, h_out, htop ? htop : h_out, b_ih, b_hh};
  for (const void* p : ptrs)
    if (!aligned16(p)) return GIC_OK;
  // units per CTA: the widest tile that still gives at least ~3/4 of the SMs a CTA
  const int mt = cdiv(B, BM);
  int U = 32;
  if ((H % 32) || (H / 32) * mt * 4 < 3 * num_sms()) U = 16;
  if (U == 16 && ((H % 16) || (H / 16) * mt * 4 < 3 * num_sms())) U = 8;
  { const int u = option("GIC_LSTM_U", 0); if ((u == 8 || u == 16 || u == 32) && H % u == 0) U = u; }   // tuning experiments
  const bool rn = tf32_round_in_tma();
  CUtensorMap tx, th, twi, twh;
  bool ok = make_map(&tx, x, B, In, In, BK, BM, rn, false) && make_map(&th, h_prev, B, H, H, BK, BM, rn, false) &&
            make_map(&twi, W_ih, 4 * H, In, In, BK, U, rn, false) && make_map(&twh, W_hh, 4 * H, H, H, BK, U, rn, false);
  if (!ok) return GIC_OK;
  static bool attr = false;
  if (!attr) {
    cudaFuncSetAttribute(lstm_step_tf32_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, LstmCfg<8>::SMEM);
    cudaFuncSetAttribute(lstm_step_tf32_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, LstmCfg<16>::SMEM);
    cudaFuncSetAttribute(lstm_step_tf32_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, LstmCfg<32>::SMEM);
    attr = true;
  }
  ProfScope prof(PROF_GEMM_DECODE, 2.0 * B * 4 * H * (In + H), stream);
  dim3 grid(H / U, mt);
  cudaError_t le;
#define GIC_LSTM(U_) le = launch_pdl(lstm_step_tf32_kernel<U_>, grid, dim3(NTHREADS), LstmCfg<U_>::SMEM, stream, tx, th, twi, twh, B, H, In, b_ih, b_hh, c_prev, acts, c_out, h_out, htop, L, t)
  if (U == 32) GIC_LSTM(32); else if (U == 16) GIC_LSTM(16); else GIC_LSTM(8);
#undef GIC_LSTM
  if (le != cudaSuccess) { set_error("lstm_step_tf32_kernel launch: %s", cudaGetErrorString(le)); return GIC_ERR_CUDA; }
  int rc = check_launch("lstm_step_tf32_kernel");
  if (rc == GIC_OK) *handled = true;
  return rc;
}

}  // namespace gic
