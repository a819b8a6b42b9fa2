// K4 (tensor cores, low-rank radial path): the fused pairwise kernel when the radial-trunk outputs of a pair,
// G = [g(e)]_e in R^{E x 128}, are numerically low rank.
//
// For distance-only radial functions (no per-edge features besides r_ij: BASELINE cfg1/2/3/5) every row of G is a point
// on a smooth one-parameter curve g(|r_ij|), and G has numerical rank ~16 to 1e-7 (measured, DESIGN.md section 4.2).
// The host factors  G ~= U V^T  (U: E x r, V: 128 x r orthonormal, residual verified every forward) and folds V into the
// last radial layer:
//     R[e,(o,i,f)] = W3[(o,i,f),:] . g[e,:] + b3  =  [U[e,:], 1] . [F'[(o,i,f),:], b3]      with F' = W3 V  (N x r)
// so the dense contraction has K = r+1 <= 64 instead of 128 and the bias rides along as one more K column.  Everything
// downstream is unchanged:   out[e,o,p] (+)= sum_{i,f} R[e,o,i,f] * T[e,i,f,p]   (reference S:294-299, 326-343, 251-254).
//
// With the GEMM 4-8x cheaper the kernel is bound by its epilogue (P fp32 FMAs per R element), so this variant is built
// around the epilogue: 16 epilogue warps (one per TMEM lane quarter x 8-channel slice), 4 per SM sub-partition, each
// keeping out[e, 8 o, P] in registers, packed fp32x2 FMAs only (no bias add), T values from conflict-free LDS.128.
//
// One CTA = 128 edges x 32 channels, loops over ceil(C_in*f/4) steps; per step one N=128 accumulator tile (column =
// if_local*32 + o_local), 3 passes (fp16 hi/lo split) x Kp/16 tcgen05.mma with A (= U tile, hi/lo) resident in tensor
// memory and B tiles (F' image, [hi | lo] x 128 rows x 64 K, SW128) streamed by TMA bulk copies, multicast over a
// 2-CTA cluster.  640 threads: warp 0 W producer, warps 1 and 3 MMA issuers (even / odd steps; warp 1 owns the TMEM allocation),
// warp 2 T producer, warps 4-19 epilogue.  (Round 2: the production path moved to csrc/zgemm.cu, DESIGN.md 4.5; this kernel
// serves fibers that are not multiples of 128 channels.)
#include "common.cuh"
#include "tc_ptx.cuh"
#include <cstdlib>
#include <algorithm>

namespace se3 {

constexpr int kLrThreads = 640;
constexpr uint32_t kLrUnitBytes = 2 * kSubBytes;   // one W tile: [hi 16 KiB | lo 16 KiB], K padded to 64
#ifndef SE3_LR_W_SLOTS
#define SE3_LR_W_SLOTS 4
#endif
#ifndef SE3_LR_T_STAGES
#define SE3_LR_T_STAGES 4
#endif
// timing experiments only (results are wrong): move only a fraction of each W unit / T stage
#ifndef SE3_LR_DBG_WDIV
#define SE3_LR_DBG_WDIV 1
#endif
#ifndef SE3_LR_DBG_TDIV
#define SE3_LR_DBG_TDIV 1
#endif
// 1: one "step" barrier pair (accumulator tile + T stage) instead of separate accumulator / T barriers: the epilogue pays one
// mbarrier wait and one arrive per step.  step_full[s % R] <- tcgen05.commit of the step's MMAs + complete_tx of its T stage
// (count 2 + tx bytes); step_empty[s % R] <- the 16 epilogue warps; the MMA warps reuse the TMEM buffer of step s-3 after
// step_empty of that step, the T producer a stage after step_empty of step s-R.
#ifndef SE3_LR_MERGED
#define SE3_LR_MERGED 0
#endif
constexpr int kLrWSlots = SE3_LR_W_SLOTS;
constexpr int kLrTStages = SE3_LR_T_STAGES;
constexpr int kLrAcc = 3;                          // TMEM accumulator buffers (the MMA -> epilogue -> MMA round trip is long)
constexpr uint32_t kLrTmemCols = 512;              // 3 accumulator buffers (384) + A hi (32) + A lo (32)
constexpr uint32_t kLrAHi = 384, kLrALo = 416;
constexpr uint32_t kLrIdesc = (1u << 4) | ((128u >> 3) << 17) | ((128u >> 4) << 24);   // fp16 x fp16 -> fp32, M128 N128

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
#ifdef SE3_LR_DBG_NOLD
#pragma unroll
  for (int i = 0; i < 8; ++i) r[i] = taddr + i;
  return;
#endif
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
}

// F'' image packer: Fp fp32 [Co*Ci*F, Kp] (columns 0..r-1 = W3 V, column r = b3, rest 0) -> per 32-channel block a row of
// 32 KiB units [hi 128 x 64 | lo 128 x 64] fp16, SW128, row = if_local*32 + o_local.  A unit holds spu = 64 / Kp (Kp = 16,
// 32: 4, 2; else 1) consecutive (i,f) steps side by side along K: step j of the unit occupies K columns [j*Kp, (j+1)*Kp),
// so the streamed bytes per step are what the MMAs read (K = Kp), not a K = 64 padded tile.
__global__ void pack_lr_kernel(const float* __restrict__ Fp, int Co, int CiF, int NU, int Kp, int spu, uint8_t* __restrict__ img) {
  const int64_t tile = blockIdx.x;
  const int ob = (int)(tile / NU), un = (int)(tile % NU);
  uint8_t* dst = img + (size_t)tile * kLrUnitBytes;
  for (int t = threadIdx.x; t < 128 * 64; t += blockDim.x) {
    const int r = t >> 6, k = t & 63;
    const int sub = k / Kp, kk = k - sub * Kp;
    const int ifb = un * spu + sub;
    const int o = ob * SE3_TILE_O + (r & 31), ifx = ifb * SE3_TILE_IF + (r >> 5);
    const float w = (sub < spu && ifx < CiF) ? Fp[((size_t)o * CiF + ifx) * Kp + kk] : 0.f;
    const __half hi = __float2half_rn(w);
    const __half lo = __float2half_rn(w - __half2float(hi));
    const uint32_t off = sw128_off(r, k);
    *reinterpret_cast<__half*>(dst + off) = hi;
    *reinterpret_cast<__half*>(dst + kSubBytes + off) = lo;
  }
}

__host__ __device__ inline int lr_steps_per_unit(int Kp) { return Kp == 16 ? 4 : Kp == 32 ? 2 : 1; }

struct LrParams {
  const float* U;          // [E, 64] fp32: columns 0..r-1 = G V, column r = 1, rest 0
  const uint8_t* w_img;
  const float* T;
  float* out;
  int64_t E;
  int Co, NIFB, n_mt, n_ob, accumulate, nk16, band_m, band_o, mma_warps, spu, NU;
  int64_t out_es;          // floats between consecutive edges of the output (Co*P for the dense [E,Co,P] layout)
  int out_os;              // floats between consecutive output channels of an edge (P for the dense layout)
  int p_off[7];            // position of the kernel's component p inside an output row
  unsigned long long* trace;   // diagnostic: per-role clock64 stamps of CTA 0 ([5 roles][64 steps][8 events]) or nullptr
};

__device__ __forceinline__ void lr_stamp(unsigned long long* trace, int role, int step, int ev) {
  if (trace != nullptr && blockIdx.x == 0 && step < 64 && (threadIdx.x & 31) == 0) trace[(role * 64 + step) * 8 + ev] = clock64();
}

// TRACE builds the diagnostic variant whose CTA 0 records clock64 stamps (tools/trace_lr.py); the production kernel has none
// (the stamps cost ~5 % even when switched off at run time, measured).
template <int P, int CSZ, bool TRACE>
__global__ void __launch_bounds__(kLrThreads, 1)
pairwise_lr_kernel(const LrParams prm) {
  const float* __restrict__ U = prm.U;
  const uint8_t* __restrict__ w_img = prm.w_img;
  const float* __restrict__ T = prm.T;
  float* __restrict__ out = prm.out;
  const int64_t E = prm.E;
  const int Co = prm.Co, NIFB = prm.NIFB, n_mt = prm.n_mt, n_ob = prm.n_ob, accumulate = prm.accumulate, nk16 = prm.nk16, spu = prm.spu, NU = prm.NU;
  constexpr int PH = (P + 3) / 4;
  constexpr uint32_t kTBytes = PH * 8192u;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* base_ptr = smem_raw + (base - raw);
  const uint32_t sW = base;                                   // + slot * kLrUnitBytes
  const uint32_t sT = sW + kLrWSlots * kLrUnitBytes;          // + stage * kTBytes
  const uint32_t sBar = sT + kLrTStages * kTBytes;
  const uint32_t bar_a_full = sBar + 0;
  const uint32_t bar_w_full = sBar + 8;
  const uint32_t bar_w_empty = bar_w_full + 8 * kLrWSlots;
  const uint32_t bar_t_full = bar_w_empty + 8 * kLrWSlots;
  const uint32_t bar_t_empty = bar_t_full + 8 * kLrTStages;
  const uint32_t bar_tm_full = bar_t_empty + 8 * kLrTStages;  // [kLrAcc]
  const uint32_t bar_tm_empty = bar_tm_full + 8 * kLrAcc;     // [kLrAcc]
  const uint32_t s_tmem_slot = bar_tm_empty + 8 * kLrAcc;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(base_ptr + (s_tmem_slot - base));

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // provably warp-uniform
  const uint32_t crank = (CSZ > 1) ? cluster_ctarank() : 0u;
  constexpr uint16_t kMask = (uint16_t)((1u << CSZ) - 1u);
  int64_t mt;
  int ob;
  bool active;
  {
    const int64_t cid = blockIdx.x / CSZ;
    const int n_mg = (n_mt + CSZ - 1) / CSZ;
    const int64_t per_band = (int64_t)prm.band_m * n_ob;
    const int64_t band = cid / per_band;
    const int64_t r = cid - band * per_band;
    const int64_t g0 = band * prm.band_m;
    const int rows = (int)min((int64_t)prm.band_m, (int64_t)n_mg - g0);
    const int go = (n_ob % prm.band_o == 0) ? prm.band_o : 1;
    const int64_t chunk = r / ((int64_t)rows * go);
    const int64_t rr = r - chunk * rows * go;
    ob = (int)(chunk * go + rr % go);
    mt = (g0 + rr / go) * CSZ + crank;
    active = mt < n_mt;
    if (!active) mt = n_mt - 1;
  }
  if (threadIdx.x == 0) {
    mbar_init(bar_a_full, 4);
    for (int s = 0; s < kLrWSlots; ++s) {
      mbar_init(bar_w_full + 8 * s, 1);
      mbar_init(bar_w_empty + 8 * s, CSZ * spu);   // every step of the unit commits once per CTA of the cluster
    }
    for (int s = 0; s < kLrTStages; ++s) {
      mbar_init(bar_t_full + 8 * s, SE3_LR_MERGED ? 2 : 1);
      mbar_init(bar_t_empty + 8 * s, 16);
    }
    for (int s = 0; s < kLrAcc; ++s) {
      mbar_init(bar_tm_full + 8 * s, 1);
      mbar_init(bar_tm_empty + 8 * s, 16);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s_tmem_slot), "r"(kLrTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  if (CSZ > 1) cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    if (warp == 0) {
      // ===================== W producer (warp-uniform loop, one elected lane issues) =====================
      const uint8_t* wsrc = w_img + (size_t)ob * NU * kLrUnitBytes;
      constexpr uint32_t kMove = kLrUnitBytes / SE3_LR_DBG_WDIV;
      constexpr uint32_t kShare = kMove / CSZ;
      for (int u = 0; u < NU; ++u) {
        const int slot = u % kLrWSlots;
        const uint32_t wph = (uint32_t)(u / kLrWSlots) & 1u;
        if constexpr (TRACE) lr_stamp(prm.trace, 3, u, 0);
        mbar_wait(bar_w_empty + 8 * slot, wph ^ 1u);
        if constexpr (TRACE) lr_stamp(prm.trace, 3, u, 1);
        if (elect_one()) {
          mbar_arrive_expect_tx(bar_w_full + 8 * slot, kMove);
          if (CSZ == 1) {
            bulk_g2s(sW + slot * kLrUnitBytes, wsrc + (size_t)u * kLrUnitBytes, kMove, bar_w_full + 8 * slot);
          } else {
            bulk_g2s_mc(sW + slot * kLrUnitBytes + crank * kShare, wsrc + (size_t)u * kLrUnitBytes + crank * kShare, kShare,
                        bar_w_full + 8 * slot, kMask);
          }
        }
        __syncwarp();
      }
    } else if (warp == 2) {
      // ===================== T producer =====================
      const uint8_t* tsrc = reinterpret_cast<const uint8_t*>(T) + (size_t)mt * NIFB * kTBytes;
      for (int s = 0; s < NIFB; ++s) {
        const int ts = s % kLrTStages;
        const uint32_t tph = (uint32_t)(s / kLrTStages) & 1u;
        if constexpr (TRACE) lr_stamp(prm.trace, 4, s, 0);
        mbar_wait(bar_t_empty + 8 * ts, tph ^ 1u);
        if constexpr (TRACE) lr_stamp(prm.trace, 4, s, 1);
        if (elect_one()) {
          mbar_arrive_expect_tx(bar_t_full + 8 * ts, kTBytes / SE3_LR_DBG_TDIV);
          bulk_g2s(sT + ts * kTBytes, tsrc + (size_t)s * kTBytes, kTBytes / SE3_LR_DBG_TDIV, bar_t_full + 8 * ts);
        }
        __syncwarp();
      }
    } else if (warp == 1 || (warp == 3 && prm.mma_warps == 2)) {
      // ===================== MMA issuer(s) (warp-uniform loop, one elected lane issues) =====================
      // One issuing warp spends ~600-900 cycles per step on its own serial chain (two mbarrier waits, the MMA issue, two
      // commits: measured with tools/trace_lr.py), which bounds the P <= 3 pairs; with two issuers, warp 1 takes the even
      // steps and warp 3 the odd ones.  Steps use different accumulator buffers, and every hand-off is an mbarrier, so the
      // order in which the two warps reach the tensor pipe does not matter.
      mbar_wait(bar_a_full, 0);
      tc_fence_after();
      const int s_first = (warp == 3) ? 1 : 0, s_stride = prm.mma_warps;
      for (int s = s_first; s < NIFB; s += s_stride) {
        const int st = s % kLrAcc;
        const uint32_t ph = (uint32_t)(s / kLrAcc) & 1u;
        const int un = s / spu, sub = s - un * spu;          // W unit and the K sub-range of this step inside it
        const int slot = un % kLrWSlots;
        const uint32_t wph = (uint32_t)(un / kLrWSlots) & 1u;
        if constexpr (TRACE) lr_stamp(prm.trace, 0, s, 0);
#if SE3_LR_MERGED
        if (s >= kLrAcc) {                      // the accumulator buffer was last used by step s - kLrAcc
          const int sp = s - kLrAcc;
          mbar_wait(bar_t_empty + 8 * (sp % kLrTStages), (uint32_t)(sp / kLrTStages) & 1u);
        }
#else
        mbar_wait(bar_tm_empty + 8 * st, ph ^ 1u);
#endif
        if constexpr (TRACE) lr_stamp(prm.trace, 0, s, 1);
        mbar_wait(bar_w_full + 8 * slot, wph);
        if constexpr (TRACE) lr_stamp(prm.trace, 0, s, 2);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)st * 128u;
        const uint32_t wbase = sW + slot * kLrUnitBytes;
        if (elect_one()) {
          uint32_t accum = 0;
          // pass 0: U_hi x F_hi   pass 1: U_lo x F_hi   pass 2: U_hi x F_lo
#pragma unroll
          for (int pass = 0; pass < 3; ++pass) {
            const uint32_t a_tmem = tmem_base + ((pass == 1) ? kLrALo : kLrAHi);
            const uint32_t b_part = (pass == 2) ? kSubBytes : 0u;
            for (int k16 = 0; k16 < nk16; ++k16) {
              const uint64_t bd = umma_desc_sw128(wbase + b_part + (sub * nk16 + k16) * 32);
#ifndef SE3_LR_DBG_NOMMA
              tc_mma_f16_ts(d_tmem, a_tmem + (uint32_t)(k16 * 8), bd, kLrIdesc, accum);
#else
              if (bd == 0x1234u) tc_mma_f16_ts(d_tmem, a_tmem + (uint32_t)(k16 * 8), bd, kLrIdesc, accum);
#endif
              accum = 1;
            }
          }
          if (CSZ == 1) tc_commit(bar_w_empty + 8 * slot);
          else tc_commit_mc(bar_w_empty + 8 * slot, kMask);
#if SE3_LR_MERGED
          tc_commit(bar_t_full + 8 * (s % kLrTStages));
#else
          tc_commit(bar_tm_full + 8 * st);
#endif
        }
        __syncwarp();
        if constexpr (TRACE) lr_stamp(prm.trace, 0, s, 4);
      }
    }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 104;");
    // ===================== epilogue warps =====================
    const int q = warp & 3;                    // TMEM lane quarter
    const int oq = (warp - 4) >> 2;            // which 8 of the 32 output channels
    const int el = q * 32 + lane;
    const uint32_t t_lane = ((uint32_t)(q * 32)) << 16;
    if (oq == 0) {
      // ---- A operand: this thread's row of U (fp32, 64 columns) -> fp16 hi / lo pairs -> tensor memory
      const int64_t eg = mt * SE3_TILE_E + el;
      const bool live = eg < E;
      const float4* urow = reinterpret_cast<const float4*>(U + (size_t)(live ? eg : 0) * 64);
#pragma unroll
      for (int c = 0; c < 2; ++c) {            // 32 k values -> 16 packed columns per chunk
        uint32_t hi[16], lo[16];
#pragma unroll
        for (int v = 0; v < 8; ++v) {
          const float4 x = live ? urow[c * 8 + v] : make_float4(0.f, 0.f, 0.f, 0.f);
          const float xs[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
          for (int h2 = 0; h2 < 2; ++h2) {
            const __half h0 = __float2half_rn(xs[2 * h2]), h1 = __float2half_rn(xs[2 * h2 + 1]);
            const __half l0 = __float2half_rn(xs[2 * h2] - __half2float(h0));
            const __half l1 = __float2half_rn(xs[2 * h2 + 1] - __half2float(h1));
            hi[v * 2 + h2] = (uint32_t)__half_as_ushort(h0) | ((uint32_t)__half_as_ushort(h1) << 16);
            lo[v * 2 + h2] = (uint32_t)__half_as_ushort(l0) | ((uint32_t)__half_as_ushort(l1) << 16);
          }
        }
        tmem_st16(tmem_base + t_lane + kLrAHi + (uint32_t)(c * 16), hi);
        tmem_st16(tmem_base + t_lane + kLrALo + (uint32_t)(c * 16), lo);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_a_full);
    }
    unsigned long long acc[4][P];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int p = 0; p < P; ++p) acc[a][p] = 0ull;

    {
    // The step loop is software pipelined at the granularity of one (i,f) slot (8 accumulator columns, PH T quads):
    // while slot c is contracted, the tcgen05.ld and the LDS of slot c+1 are in flight (tcgen05.wait::ld waits for every
    // outstanding load, so it is placed after the FMAs of the current slot).
    const uint32_t tcol0 = tmem_base + t_lane + (uint32_t)(oq * 8);
    const float4* Tsm = reinterpret_cast<const float4*>(base_ptr + (sT - base)) + el;
    auto contract = [&](const uint32_t (&r)[8], const float4 (&t)[PH]) {
#ifdef SE3_LR_DBG_NOFMA
      {
        unsigned long long x = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i) x ^= r[i];
#pragma unroll
        for (int h4 = 0; h4 < PH; ++h4) x ^= __float_as_uint(t[h4].x) ^ __float_as_uint(t[h4].w);
        acc[0][0] ^= x;
        return;
      }
#endif
      float tv[PH * 4];
#pragma unroll
      for (int h4 = 0; h4 < PH; ++h4) { tv[h4 * 4 + 0] = t[h4].x; tv[h4 * 4 + 1] = t[h4].y; tv[h4 * 4 + 2] = t[h4].z; tv[h4 * 4 + 3] = t[h4].w; }
#pragma unroll
      for (int p = 0; p < P; ++p) {
        const unsigned long long t2 = pack2(tv[p], tv[p]);
#pragma unroll
        for (int a = 0; a < 4; ++a)
          acc[a][p] = fma2(pack2(__uint_as_float(r[2 * a]), __uint_as_float(r[2 * a + 1])), t2, acc[a][p]);
      }
    };
    auto load_t = [&](float4 (&t)[PH], int stage, int ifl) {
#pragma unroll
      for (int h4 = 0; h4 < PH; ++h4) {
#ifdef SE3_LR_DBG_HALFLDS
        if (h4 > 0) { t[h4] = make_float4(t[0].y, t[0].x, t[0].w, t[0].z); continue; }
#endif
#ifdef SE3_LR_DBG_NOLDS
        { const float f = __int_as_float(0x3f800000 + stage + ifl); t[h4] = make_float4(f, f, f, f); continue; }
#endif
        t[h4] = Tsm[(size_t)stage * (kTBytes / 16) + (ifl * PH + h4) * 128];
      }
    };
    uint32_t ra[8], rb[8];
    float4 ta[PH], tb[PH];
#if SE3_LR_MERGED
    mbar_wait(bar_t_full, 0);
    tc_fence_after();
    tmem_ld8(tcol0, ra);
#else
    mbar_wait(bar_tm_full, 0);
    tc_fence_after();
    tmem_ld8(tcol0, ra);
    mbar_wait(bar_t_full, 0);
#endif
    load_t(ta, 0, 0);
    tmem_ld_wait();
#ifndef SE3_LR_PROBE
#define SE3_LR_PROBE 0     // measured: early try_wait probes are 0-3 % slower (same-box A/B), kept for experiments
#endif
    constexpr bool kProbe = SE3_LR_PROBE && (P >= 5);
    // running ring indices / phase parities of the current step (no div/mod in the loop)
    int st = 0, ts = 0;
    uint32_t ph_acc = 0, ph_t = 0;
    for (int s = 0; s < NIFB; ++s) {
      const uint32_t tcol = tcol0 + (uint32_t)(st * 128);
      const int trole = (warp == 4) ? 1 : (warp == 19) ? 2 : -1;
      if constexpr (TRACE) if (trole > 0) lr_stamp(prm.trace, trole, s, 0);
      // slot 0
      tmem_ld8(tcol + 32u, rb);
      load_t(tb, ts, 1);
      contract(ra, ta);
      tmem_ld_wait();
      // slot 1
      tmem_ld8(tcol + 64u, ra);
      load_t(ta, ts, 2);
      contract(rb, tb);
      tmem_ld_wait();
      int st1 = st + 1, ts1 = ts + 1;
      uint32_t pa1 = ph_acc, pt1 = ph_t;
      if (st1 == kLrAcc) { st1 = 0; pa1 ^= 1u; }
      if (ts1 == kLrTStages) { ts1 = 0; pt1 ^= 1u; }
      const bool more = s + 1 < NIFB;
      // slot 2
      tmem_ld8(tcol + 96u, rb);
      load_t(tb, ts, 3);
      // Epilogue-bound pairs (P >= 5): the next step's accumulator and T stage were completed long ago, but an
      // mbarrier.try_wait still takes ~90-190 cycles to answer; ask now and read the answers after this slot's FMAs.
      uint32_t ok_acc = 0, ok_t = 0;
      if constexpr (kProbe) {
        if (more) {
          ok_acc = mbar_try_wait(bar_tm_full + 8 * st1, pa1);
          ok_t = mbar_try_wait(bar_t_full + 8 * ts1, pt1);
        }
      }
      contract(ra, ta);
      tmem_ld_wait();
      if constexpr (TRACE) if (trole > 0) lr_stamp(prm.trace, trole, s, 1);
      // every accumulator column of this step is in registers: hand the buffer back to the MMA warp
      tc_fence_before();
      __syncwarp();
#if SE3_LR_MERGED
      // (the LDS of the last slot have been issued and the arrive is a release: the T stage goes back with the accumulator)
      if (lane == 0) mbar_arrive(bar_t_empty + 8 * ts);
#else
      if (lane == 0) mbar_arrive(bar_tm_empty + 8 * st);
#endif
      if constexpr (TRACE) if (trole > 0) lr_stamp(prm.trace, trole, s, 2);
      // slot 3, with slot 0 of the next step in flight
      if (more) {
#if SE3_LR_MERGED
        mbar_wait(bar_t_full + 8 * ts1, pt1);
#else
        if (!ok_acc) mbar_wait(bar_tm_full + 8 * st1, pa1);
#endif
        tc_fence_after();
        if constexpr (TRACE) if (trole > 0) lr_stamp(prm.trace, trole, s, 3);
        tmem_ld8(tcol0 + (uint32_t)(st1 * 128), ra);
#if !SE3_LR_MERGED
        if (!ok_t) mbar_wait(bar_t_full + 8 * ts1, pt1);
#endif
        if constexpr (TRACE) if (trole > 0) lr_stamp(prm.trace, trole, s, 4);
        load_t(ta, ts1, 0);
      }
      contract(rb, tb);
      if (more) tmem_ld_wait();
      __syncwarp();
#if !SE3_LR_MERGED
      if (lane == 0) mbar_arrive(bar_t_empty + 8 * ts);
#endif
      if constexpr (TRACE) if (trole > 0) lr_stamp(prm.trace, trole, s, 5);
      st = st1; ts = ts1; ph_acc = pa1; ph_t = pt1;
    }
    }
    // write out[e, ob*32 + oq*8 + (0..7), 0..P)
    const int64_t e = mt * SE3_TILE_E + el;
    if (active && e < E) {
      const int ld = prm.out_os;
      float* dst = out + (size_t)e * prm.out_es + (size_t)(ob * SE3_TILE_O + oq * 8) * ld;
      // read-modify-write in two phases (all loads of a batch, then all stores): with run-time strides the compiler has to
      // assume that a store may alias the next load, and a load -> store -> load chain costs one DRAM round trip per value
      // (measured: +3.7 ms on a 2.5 ms launch)
      constexpr int AB = (P <= 3) ? 4 : 1;             // channel pairs per batch (register budget)
#pragma unroll
      for (int a0 = 0; a0 < 4; a0 += AB) {
        float prev[AB][P][2];
#pragma unroll
        for (int a = 0; a < AB; ++a)
#pragma unroll
          for (int p = 0; p < P; ++p) {
            const float* d0 = dst + (2 * (a0 + a)) * ld + prm.p_off[p];
            prev[a][p][0] = accumulate ? __ldcg(d0) : 0.f;
            prev[a][p][1] = accumulate ? __ldcg(d0 + ld) : 0.f;
          }
#pragma unroll
        for (int a = 0; a < AB; ++a)
#pragma unroll
          for (int p = 0; p < P; ++p) {
            float v0, v1;
            unpack2(acc[a0 + a][p], v0, v1);
            float* d0 = dst + (2 * (a0 + a)) * ld + prm.p_off[p];
            d0[0] = v0 + prev[a][p][0];
            d0[ld] = v1 + prev[a][p][1];
          }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (CSZ > 1) cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kLrTmemCols) : "memory");
  }
}

template <int P>
static size_t lr_smem_bytes() {
  constexpr int PH = (P + 3) / 4;
  return 1024 + kLrWSlots * kLrUnitBytes + kLrTStages * (PH * 8192u) + 256;
}

template <int P, int CSZ, bool TRACE>
static int launch_lr(const LrParams& prm, cudaStream_t s) {
  const size_t smem = lr_smem_bytes<P>();
  auto kern = pairwise_lr_kernel<P, CSZ, TRACE>;
  SE3_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int n_mg = (prm.n_mt + CSZ - 1) / CSZ;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)((int64_t)n_mg * prm.n_ob * CSZ));
  cfg.blockDim = dim3(kLrThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CSZ;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  SE3_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, prm));
  return SE3_OK;
}

static int lr_env_int(const char* name, int dflt) {
  const char* v = getenv(name);
  return v ? atoi(v) : dflt;
}

}  // namespace se3

extern "C" int64_t se3_lowrank_image_bytes(int Co, int Ci, int F, int Kp) {
  if (Co <= 0 || Ci <= 0 || F <= 0 || Co % SE3_TILE_O != 0 || Kp < 16 || Kp > 64 || Kp % 16 != 0) return -1;
  const int64_t NIFB = se3::ceil_div((int64_t)Ci * F, SE3_TILE_IF);
  const int64_t NU = se3::ceil_div(NIFB, (int64_t)se3::lr_steps_per_unit(Kp));
  return (int64_t)(Co / SE3_TILE_O) * NU * se3::kLrUnitBytes;
}

extern "C" int se3_pack_lowrank(const float* Fp, int Co, int Ci, int F, int Kp, void* image, void* stream) {
  using namespace se3;
  SE3_REQUIRE(Co > 0 && Ci > 0 && F > 0 && Co % SE3_TILE_O == 0, "se3_pack_lowrank: Co must be a positive multiple of %d", SE3_TILE_O);
  SE3_REQUIRE(Kp >= 16 && Kp <= 64 && Kp % 16 == 0, "se3_pack_lowrank: Kp=%d must be 16, 32, 48 or 64", Kp);
  const int CiF = Ci * F;
  const int NIFB = (int)ceil_div(CiF, SE3_TILE_IF);
  const int spu = lr_steps_per_unit(Kp);
  const int NU = (int)ceil_div(NIFB, spu);
  const int64_t tiles = (int64_t)(Co / SE3_TILE_O) * NU;
  SE3_REQUIRE(tiles < 2147483647ll, "se3_pack_lowrank: too many tiles");
  pack_lr_kernel<<<(unsigned)tiles, 256, 0, as_stream(stream)>>>(Fp, Co, CiF, NU, Kp, spu, reinterpret_cast<uint8_t*>(image));
  SE3_LAUNCH_OK();
  return SE3_OK;
}

static int pairwise_lr_impl(const float* U, const void* w_img, const float* T, int64_t E, int Co, int Ci, int F, int P, int Kp,
                            int accumulate, float* out, int64_t out_es, int out_os, const int* p_off, unsigned long long* trace, void* stream) {
  using namespace se3;
  SE3_REQUIRE(E > 0 && Co > 0 && Ci > 0 && F > 0, "se3_pairwise_lr_fwd: bad sizes");
  SE3_REQUIRE(Co % SE3_TILE_O == 0, "se3_pairwise_lr_fwd: Co=%d must be a multiple of %d", Co, SE3_TILE_O);
  SE3_REQUIRE(P == 1 || P == 2 || P == 3 || P == 5 || P == 7, "se3_pairwise_lr_fwd: P=%d unsupported (1, 2, 3, 5, 7)", P);
  SE3_REQUIRE(out_es > 0 && out_os > 0, "se3_pairwise_lr_fwd: bad output strides");
  SE3_REQUIRE(Kp >= 16 && Kp <= 64 && Kp % 16 == 0, "se3_pairwise_lr_fwd: Kp=%d must be 16, 32, 48 or 64", Kp);
  SE3_REQUIRE((ceil_div(E, SE3_TILE_E) + 4) * (Co / SE3_TILE_O) < 2147483647ll, "se3_pairwise_lr_fwd: grid too large");
  LrParams prm;
  prm.U = U;
  prm.w_img = reinterpret_cast<const uint8_t*>(w_img);
  prm.T = T;
  prm.out = out;
  prm.E = E;
  prm.Co = Co;
  prm.NIFB = (int)ceil_div((int64_t)Ci * F, SE3_TILE_IF);
  prm.n_mt = (int)ceil_div(E, SE3_TILE_E);
  prm.n_ob = Co / SE3_TILE_O;
  prm.accumulate = accumulate;
  prm.nk16 = Kp / 16;
  prm.out_es = out_es;
  prm.out_os = out_os;
  for (int p = 0; p < 7; ++p) prm.p_off[p] = (p < P) ? (p_off ? p_off[p] : p) : 0;
  for (int p = 0; p < P; ++p)
    SE3_REQUIRE(prm.p_off[p] >= 0 && prm.p_off[p] < out_es, "se3_pairwise_lr_fwd: p_off[%d]=%d outside the edge row", p, prm.p_off[p]);
  prm.spu = lr_steps_per_unit(Kp);
  prm.NU = (int)ceil_div((int64_t)prm.NIFB, (int64_t)prm.spu);
  prm.trace = trace;
  prm.mma_warps = lr_env_int("SE3B200_LR_MMA_WARPS", 2) == 1 ? 1 : 2;
  const int csz = (trace == nullptr && lr_env_int("SE3B200_LR_CLUSTER", 2) == 1) ? 1 : 2;
  prm.band_o = std::max(1, lr_env_int("SE3B200_LR_BANDO", 4));
  prm.band_m = std::max(1, 148 / (csz * prm.band_o));
  cudaStream_t s = as_stream(stream);
#define SE3_LR_CASE(PP) (trace != nullptr ? launch_lr<PP, 2, true>(prm, s) : csz == 1 ? launch_lr<PP, 1, false>(prm, s) : launch_lr<PP, 2, false>(prm, s))
  switch (P) {
    case 1: return SE3_LR_CASE(1);
    case 2: return SE3_LR_CASE(2);
    case 3: return SE3_LR_CASE(3);
    case 5: return SE3_LR_CASE(5);
    default: return SE3_LR_CASE(7);
  }
#undef SE3_LR_CASE
}

extern "C" int se3_pairwise_lr_fwd(const float* U, const void* w_img, const float* T, int64_t E, int Co, int Ci, int F, int P,
                                   int Kp, int accumulate, float* out, void* stream) {
  return pairwise_lr_impl(U, w_img, T, E, Co, Ci, F, P, Kp, accumulate, out, (int64_t)Co * P, P, nullptr, nullptr, stream);
}

// Diagnostic (tools/ only): same launch, and CTA 0 records clock64 stamps of its warp roles into trace[5][64][8].
extern "C" int se3_pairwise_lr_trace(const float* U, const void* w_img, const float* T, int64_t E, int Co, int Ci, int F, int P,
                                     int Kp, int accumulate, float* out, unsigned long long* trace, void* stream) {
  return pairwise_lr_impl(U, w_img, T, E, Co, Ci, F, P, Kp, accumulate, out, (int64_t)Co * P, P, nullptr, trace, stream);
}
