// Backward of the spatial self-attention (csrc/spatial_attn_tc.cu) on tcgen05 tensor cores with TMEM accumulators and
// tensor-map TMA operand loads, sm_100a: the autograd of the xformers seam (reference models/attention.py:535-542) that
// torch.autograd.grad traverses at utils/motionclone_functions.py:236.
//
// With P = softmax(scale S), S = Q K^T, D_r = sum_e dO_re O_re:
//     dV = P^T dO      dP = dO V^T      dS = scale * P o (dP - D)      dQ = dS K      dK = dS^T Q
// P is recomputed from the forward's log-sum-exp (no N x N tensor is ever stored). Three launches:
//   prep       : lse2 = lse * log2(e) and Dsc = scale * D per (frame, head, token), padded to a multiple of 64 tokens
//   dQ kernel  : CTA = 128 queries, streams 64-key tiles:   S, dP (M=128 q, N=64 keys) -> dS -> smem -> dQ += dS K
//   dKV kernel : CTA = 128 keys,   streams 64-query tiles:  S^T = K Q^T, dP^T = V dO^T (M=128 keys, N=64 q)
//                -> P^T, dS^T -> smem -> dV += P^T dO, dK += dS^T Q
// Both kernels: 8 compute warps (thread = TMEM lane = tile row, the two warps that share a lane quarter split the 64
// columns) + an MMA warp and a TMA warp (one thread each: MMA issue never waits behind a ring refill); accumulators in TMEM; 2 CTAs per SM where the
// TMEM budget allows. Every streamed [rows][DH] tile serves two GEMMs through two descriptors - K-major where DH is
// contracted (S, dP), MN-major where the rows are (dS K, P^T dO, dS^T Q) - so nothing is transposed or copied twice.
// The tiles the threads produce (dS, P^T, dS^T) never touch shared memory: they go back into tensor memory as fp16 pairs
// (tcgen05.st) and are the A operands of the next MMAs (tcgen05.mma with A in TMEM); for head dims <= 48 the resident
// operand tiles (Q, dO in the dQ kernel, V in the dK/dV kernel) are moved into tensor memory once, too. An MMA whose A
// operand comes from shared memory re-reads 4 KB of it per k16 step - that traffic, not the math, bounded the first
// version (ncu: tensor pipe 47-52 % busy at ~70 cycles per MMA). There are no
// masks: rows past the end of the sequence are zero-filled by the TMA unit, and a zero K / V / Q / dO row contributes
// nothing to any of the sums (the padded statistics keep every intermediate finite). The two-kernel split recomputes S and
// dP once more than a fused kernel would but needs no atomics on dQ: results are deterministic.
#include <math.h>

#include "tma_common.cuh"

namespace mc {

constexpr int kBM = 128;         // resident rows per CTA (UMMA M)
constexpr int kBT = 64;          // streamed tile height (keys in the dQ kernel, queries in the dKV kernel)
constexpr int kBComputeWarps = 8;
constexpr int kBMmaWarp = kBComputeWarps, kBTmaWarp = kBComputeWarps + 1;  // lane 0 of each: MMA issue / TMA loads
constexpr int kBThreads = (kBComputeWarps + 2) * 32;

struct FABwdParams {
  const float* lse2;   // [B][H][Npad]  lse * log2(e)      (padding: 0)
  const float* dsc;    // [B][H][Npad]  scale * rowsum(dO o O)   (padding: 0)
  __half *dq, *dk, *dv;
  int64_t g_sb, g_sr;  // dq / dk / dv share one stride pattern (column blocks of one fused gradient buffer, or separate)
  int B, N, H, Npad;
  float scale, scale_log2e;
};

// lse2[b][h][r] = lse * log2 e;  dsc[b][h][r] = scale * sum_e dO[b][r][h][e] * O[b][r][h][e];  zeros for N <= r < Npad
template <int DH>
__global__ void __launch_bounds__(256) attn_bwd_prep_kernel(const __half* __restrict__ o, const __half* __restrict__ d_o,
                                                            const float* __restrict__ lse, float* __restrict__ lse2,
                                                            float* __restrict__ dsc, int64_t o_sb, int64_t o_sr,
                                                            int64_t do_sb, int64_t do_sr, int B, int N, int Npad, int H,
                                                            float scale) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // ((b * Npad) + r) * H + h
  if (i >= (int64_t)B * Npad * H) return;
  const int h = (int)(i % H);
  const int64_t br = i / H;
  const int r = (int)(br % Npad), b = (int)(br / Npad);
  const int64_t dst = ((int64_t)b * H + h) * Npad + r;
  if (r >= N) {
    lse2[dst] = 0.f, dsc[dst] = 0.f;
    return;
  }
  const uint4* po = reinterpret_cast<const uint4*>(o + b * o_sb + (int64_t)r * o_sr + h * DH);
  const uint4* pd = reinterpret_cast<const uint4*>(d_o + b * do_sb + (int64_t)r * do_sr + h * DH);
  float acc = 0.f;
#pragma unroll
  for (int c = 0; c < DH / 8; ++c) {
    const uint4 a = po[c], g = pd[c];
    const __half2* ah = reinterpret_cast<const __half2*>(&a);
    const __half2* gh = reinterpret_cast<const __half2*>(&g);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 x = __half22float2(ah[j]), y = __half22float2(gh[j]);
      acc = fmaf(x.x, y.x, acc);
      acc = fmaf(x.y, y.y, acc);
    }
  }
  lse2[dst] = lse[((int64_t)b * H + h) * N + r] * 1.44269504088896340736f;
  dsc[dst] = acc * scale;
}

// D[128 x 64] = A[128 x DH] B[64 x DH]^T (S, dP, S^T, dP^T) with B a 64-row tile (K-major) and A resident in tensor memory
// (head dims <= 48: DHP / 2 packed columns at a_tmem, see smem_row_to_tmem); an A tile in shared memory takes issue_kmajor
template <int DH>
__device__ __forceinline__ void issue_qk64_ts(uint32_t d_tmem, uint32_t a_tmem, uint32_t sB) {
  using TB = TileParts<DH, kBT>;
  static_assert(TB::N64 == 1 && TB::N16 == 0, "tensor-memory A operands: head dims <= 48");
  const uint32_t idesc = umma_idesc_f16(128, kBT, false, false);
#pragma unroll
  for (int ks = 0; ks < TB::KS64; ++ks) umma_f16_ts(d_tmem, a_tmem + ks * 8, desc_k128(sB, ks), idesc, ks > 0 ? 1u : 0u);
}

template <int DH>
struct FABwdCfg {
  using TA = TileParts<DH, 128>;   // resident tiles
  using TB = TileParts<DH, kBT>;   // streamed tiles
  static constexpr int DHP = TA::DHP;
  static constexpr bool AT = DHP <= 48;   // resident operand tiles live in tensor memory as A operands
  static constexpr int KP = DHP / 2;      // packed columns of a resident [128][DHP] fp16 tile
  // Streamed-tile ring depth. A stage is refilled when the MMAs that read it have completed, i.e. NS - 1 tiles before it is
  // needed again: with 2 stages the TMA round trip (~1 us) sat on the critical path of every tile (round-2 ncu: 58 % of
  // stall samples were warps parked on mbarriers with the tensor pipe half idle).
  static constexpr int NS = DHP <= 48 ? 4 : (DHP <= 80 ? 3 : 2);
  // dQ kernel. shared memory: Q, dO (only staging when AT); K, V ring.
  static constexpr int DQ_OFF_Q = 0, DQ_OFF_DO = TA::BYTES, DQ_OFF_K = 2 * TA::BYTES, DQ_OFF_V = DQ_OFF_K + NS * TB::BYTES;
  static constexpr int DQ_OFF_BAR = DQ_OFF_V + NS * TB::BYTES, DQ_SMEM = DQ_OFF_BAR + 256 + 1024;
  // tensor memory: S [0,64) dP [64,128) dS(fp16 pairs) [128,160) dQ [160,160+DHP) [Q, dO packed when AT]
  static constexpr int DQ_DS = 128, DQ_ACC = 160, DQ_QT = 160 + DHP, DQ_DOT = DQ_QT + KP;
  static constexpr int DQ_NEED = AT ? DQ_DOT + KP : DQ_ACC + DHP;
  static constexpr int DQ_TCOLS = DQ_NEED <= 256 ? 256 : 512;
  static constexpr int DQ_CTAS = ctas_per_sm(DQ_TCOLS, DQ_SMEM);
  // dKV kernel. shared memory: K, V resident; Q, dO double-buffered.
  static constexpr int KV_OFF_K = 0, KV_OFF_V = TA::BYTES, KV_OFF_Q = 2 * TA::BYTES, KV_OFF_DO = KV_OFF_Q + NS * TB::BYTES;
  // per-query statistics of the streamed tile ride the same ring: 64 x (lse2, scale D) fp32 = 512 B per stage
  static constexpr int KV_OFF_BAR = KV_OFF_DO + NS * TB::BYTES, KV_OFF_ST = KV_OFF_BAR + 256;
  static constexpr int KV_SMEM = KV_OFF_ST + NS * 512 + 1024;
  // tensor memory: S^T [0,64) dP^T [64,128) (P^T / dS^T are written back over them as fp16 pairs) dV, dK [V packed when AT]
  static constexpr int DV_COL = 128, DK_COL = 128 + DHP, KV_VT = 128 + 2 * DHP;
  static constexpr int KV_NEED = AT ? KV_VT + KP : KV_VT;
  static constexpr int KV_TCOLS = KV_NEED <= 256 ? 256 : 512;
  static constexpr int KV_CTAS = ctas_per_sm(KV_TCOLS, KV_SMEM);
};

// half a TMEM row (columns [c0, c0 + ncol) of DHP fp32) -> fp16 -> global
template <int DH>
__device__ __forceinline__ void store_cols_from_tmem(uint32_t taddr, __half* grow, bool valid, int c0, int ncol) {
  for (int cc = c0; cc < c0 + ncol; cc += 16) {
    uint32_t r[16];
    tmem_ld16(taddr + cc, r);
    tmem_ld_wait();
    if (valid) {
#pragma unroll
      for (int half8 = 0; half8 < 2; ++half8) {
        if (cc + half8 * 8 < DH) {
          uint4 pk;
          pk.x = pack_half2(__uint_as_float(r[half8 * 8 + 0]), __uint_as_float(r[half8 * 8 + 1]));
          pk.y = pack_half2(__uint_as_float(r[half8 * 8 + 2]), __uint_as_float(r[half8 * 8 + 3]));
          pk.z = pack_half2(__uint_as_float(r[half8 * 8 + 4]), __uint_as_float(r[half8 * 8 + 5]));
          pk.w = pack_half2(__uint_as_float(r[half8 * 8 + 6]), __uint_as_float(r[half8 * 8 + 7]));
          *reinterpret_cast<uint4*>(grow + cc + half8 * 8) = pk;
        }
      }
    }
  }
}

// columns of the DHP-wide accumulator owned by column-half `hh` of a row (multiples of 16)
template <int DHP>
__device__ __forceinline__ void half_cols(int hh, int& c0, int& ncol) {
  constexpr int FIRST = ((DHP / 16 + 1) / 2) * 16;
  c0 = hh == 0 ? 0 : FIRST;
  ncol = hh == 0 ? FIRST : DHP - FIRST;
}

// ------------------------------------------------ dQ ------------------------------------------------------------------
template <int DH>
__global__ void __launch_bounds__(kBThreads, FABwdCfg<DH>::DQ_CTAS)
spatial_attn_bwd_dq_kernel(const __grid_constant__ CUtensorMap mq128, const __grid_constant__ CUtensorMap mq32,
                           const __grid_constant__ CUtensorMap mdo128, const __grid_constant__ CUtensorMap mdo32,
                           const __grid_constant__ CUtensorMap mk128, const __grid_constant__ CUtensorMap mk32,
                           const __grid_constant__ CUtensorMap mv128, const __grid_constant__ CUtensorMap mv32,
                           const FABwdParams prm) {
  using X = FABwdCfg<DH>;
  using TA = typename X::TA;
  using TB = typename X::TB;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sQ = smem + X::DQ_OFF_Q;
  uint8_t* sDO = smem + X::DQ_OFF_DO;
  uint8_t* sK = smem + X::DQ_OFF_K;   // NS stages
  uint8_t* sV = smem + X::DQ_OFF_V;   // NS stages
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + X::DQ_OFF_BAR);
  uint64_t* bar_q = bars + 0;        // Q and dO landed
  uint64_t* sdp_full = bars + 1;     // S_j, dP_j in TMEM
  uint64_t* sdp_free = bars + 2;     // copied to registers (8 warp arrivals)
  uint64_t* ds_full = bars + 3;      // dS_j in TMEM (8 warp arrivals)
  uint64_t* dq_done = bars + 4;      // dQ += dS_j K_j completed
  uint64_t* a_ready = bars + 5;      // Q, dO copied into tensor memory (8 warp arrivals; AT only)
  uint64_t* bar_kv = bars + 8;       // [NS] K_j, V_j landed in stage j % NS
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8 + X::NS);
  constexpr int NS = X::NS;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int qt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int q0 = qt * kBM, N = prm.N;
  const int T_tiles = (N + kBT - 1) / kBT;

  if (warp == kBMmaWarp) {
    tmem_alloc<X::DQ_TCOLS>(tmem_slot);
    if (lane == 0) {
      mbar_init(bar_q, 1), mbar_init(sdp_full, 1);
      mbar_init(sdp_free, kBComputeWarps), mbar_init(ds_full, kBComputeWarps), mbar_init(dq_done, 1);
      mbar_init(a_ready, kBComputeWarps);
      for (int i = 0; i < NS; ++i) mbar_init(bar_kv + i, 1);
      fence_mbar_init();
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == kBTmaWarp) {
    // ---- TMA warp: resident tiles, then the K / V ring (a stage is refilled as soon as the MMAs that read it are done) ----
    if (lane == 0) {
      mbar_arrive_expect_tx(bar_q, 2 * TA::BYTES);
      tma_load_tile<DH, 128>(sQ, &mq128, &mq32, bar_q, q0, h, b);
      tma_load_tile<DH, 128>(sDO, &mdo128, &mdo32, bar_q, q0, h, b);
      for (int j = 0; j < NS && j < T_tiles; ++j) {
        mbar_arrive_expect_tx(bar_kv + j, 2 * TB::BYTES);
        tma_load_tile<DH, kBT>(sK + j * TB::BYTES, &mk128, &mk32, bar_kv + j, j * kBT, h, b);
        tma_load_tile<DH, kBT>(sV + j * TB::BYTES, &mv128, &mv32, bar_kv + j, j * kBT, h, b);
      }
      for (int j = 0; j + NS < T_tiles; ++j) {
        const int st = j % NS;
        mbar_wait(dq_done, j & 1);  // K_j / V_j consumed
        mbar_arrive_expect_tx(bar_kv + st, 2 * TB::BYTES);
        tma_load_tile<DH, kBT>(sK + st * TB::BYTES, &mk128, &mk32, bar_kv + st, (j + NS) * kBT, h, b);
        tma_load_tile<DH, kBT>(sV + st * TB::BYTES, &mv128, &mv32, bar_kv + st, (j + NS) * kBT, h, b);
      }
    }
  } else if (warp == kBMmaWarp) {
    // ---- MMA warp: one thread issues every tcgen05.mma ----
    if (lane == 0) {
      auto issue_sdp = [&](int stage) {
        if constexpr (X::AT) {
          issue_qk64_ts<DH>(tmem_base, tmem_base + X::DQ_QT, smem_u32(sK + stage * TB::BYTES));
          issue_qk64_ts<DH>(tmem_base + 64, tmem_base + X::DQ_DOT, smem_u32(sV + stage * TB::BYTES));
        } else {
          issue_kmajor<DH, kBM, kBT>(tmem_base, smem_u32(sQ), smem_u32(sK + stage * TB::BYTES));
          issue_kmajor<DH, kBM, kBT>(tmem_base + 64, smem_u32(sDO), smem_u32(sV + stage * TB::BYTES));
        }
      };
      if constexpr (X::AT) mbar_wait(a_ready, 0);
      else mbar_wait(bar_q, 0);
      mbar_wait(bar_kv, 0);
      tc_fence_after();
      issue_sdp(0);
      umma_commit(sdp_full);
      for (int j = 0; j < T_tiles; ++j) {
        const uint32_t ph = j & 1;
        const int st = j % NS;
        if (j + 1 < T_tiles) {
          const int sn = (j + 1) % NS;
          mbar_wait(bar_kv + sn, ((j + 1) / NS) & 1);
          mbar_wait(sdp_free, ph);
          tc_fence_after();
          issue_sdp(sn);
          umma_commit(sdp_full);
        }
        mbar_wait(ds_full, ph);
        tc_fence_after();
        issue_ts_mn<DH, kBT>(tmem_base + X::DQ_ACC, [&](int ks) { return tmem_base + X::DQ_DS + ks * 8; },
                             smem_u32(sK + st * TB::BYTES), j > 0);
        umma_commit(dq_done);
      }
    }
  } else {
    const int rq = warp & 3, hh = warp >> 2;  // TMEM lane quarter, column half
    const int r = rq * 32 + lane;             // tile row = TMEM lane
    const uint32_t lane_addr = tmem_base + ((uint32_t)(rq * 32) << 16);
    if constexpr (X::AT) {  // Q (column half 0) and dO (column half 1) rows -> tensor memory, once
      mbar_wait(bar_q, 0);
      smem_row_to_tmem<X::DHP>(hh == 0 ? sQ : sDO, r, lane_addr + (hh == 0 ? X::DQ_QT : X::DQ_DOT));
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(a_ready);
    }
    const int row = q0 + r;
    const bool rvalid = row < N;
    const int64_t srow = ((int64_t)b * prm.H + h) * prm.Npad + (rvalid ? row : 0);
    const float nl2 = -prm.lse2[srow];
    const float nD = -prm.dsc[srow];
    const float c = prm.scale_log2e, sc = prm.scale;
    for (int j = 0; j < T_tiles; ++j) {
      const uint32_t ph = j & 1;
      mbar_wait(sdp_full, ph);
      tc_fence_after();
      uint32_t s[32], dp[32];
      tmem_ld32(lane_addr + hh * 32, s);
      tmem_ld32(lane_addr + 64 + hh * 32, dp);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(sdp_free);
#pragma unroll
      for (int i = 0; i < 32; i += 2) {  // dS = P o (scale dP - scale D)
        float p0, p1;
        ex2_pair(i >> 1, __uint_as_float(s[i]), __uint_as_float(s[i + 1]), c, nl2, p0, p1);
        s[i >> 1] = pack_half2(p0 * fmaf(__uint_as_float(dp[i]), sc, nD), p1 * fmaf(__uint_as_float(dp[i + 1]), sc, nD));
      }
      if (j > 0) {
        mbar_wait(dq_done, ph ^ 1);  // dS_{j-1} consumed by its MMA
        tc_fence_after();
      }
      tmem_st16(lane_addr + X::DQ_DS + hh * 16, s);  // keys [32 hh, 32 hh + 32) = packed columns [16 hh, 16 hh + 16)
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(ds_full);
    }
    mbar_wait(dq_done, (T_tiles - 1) & 1);
    tc_fence_after();
    int c0, ncol;
    half_cols<X::DHP>(hh, c0, ncol);
    store_cols_from_tmem<DH>(lane_addr + X::DQ_ACC, prm.dq + (int64_t)b * prm.g_sb + (int64_t)row * prm.g_sr + h * DH, rvalid,
                             c0, ncol);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kBMmaWarp) {
    __syncwarp();
    tmem_dealloc<X::DQ_TCOLS>(tmem_base);
  }
}

// ------------------------------------------------ dK, dV --------------------------------------------------------------
template <int DH>
__global__ void __launch_bounds__(kBThreads, FABwdCfg<DH>::KV_CTAS)
spatial_attn_bwd_dkv_kernel(const __grid_constant__ CUtensorMap mk128, const __grid_constant__ CUtensorMap mk32,
                            const __grid_constant__ CUtensorMap mv128, const __grid_constant__ CUtensorMap mv32,
                            const __grid_constant__ CUtensorMap mq128, const __grid_constant__ CUtensorMap mq32,
                            const __grid_constant__ CUtensorMap mdo128, const __grid_constant__ CUtensorMap mdo32,
                            const FABwdParams prm) {
  using X = FABwdCfg<DH>;
  using TA = typename X::TA;
  using TB = typename X::TB;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sK = smem + X::KV_OFF_K;
  uint8_t* sV = smem + X::KV_OFF_V;
  uint8_t* sQ = smem + X::KV_OFF_Q;    // NS stages
  uint8_t* sDO = smem + X::KV_OFF_DO;  // NS stages
  uint8_t* sST = smem + X::KV_OFF_ST;  // NS stages of [64 lse2 | 64 scale D]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + X::KV_OFF_BAR);
  uint64_t* bar_kv = bars + 0;      // K, V landed
  uint64_t* st_full = bars + 1;     // S^T_i, dP^T_i in TMEM
  uint64_t* pt_full = bars + 2;     // P^T_i, dS^T_i written back to TMEM, S^T_i / dP^T_i consumed (8 warp arrivals)
  uint64_t* dkv_done = bars + 3;    // dV, dK updates of tile i completed
  uint64_t* a_ready = bars + 4;     // V copied into tensor memory (4 warp arrivals; AT only)
  uint64_t* bar_q = bars + 8;       // [NS] Q_i, dO_i landed in stage i % NS
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8 + X::NS);
  constexpr int NS = X::NS;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int kt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int k0 = kt * kBM, N = prm.N;
  const int T_tiles = (N + kBT - 1) / kBT;

  if (warp == kBMmaWarp) {
    tmem_alloc<X::KV_TCOLS>(tmem_slot);
    if (lane == 0) {
      mbar_init(bar_kv, 1), mbar_init(st_full, 1);
      mbar_init(pt_full, kBComputeWarps), mbar_init(dkv_done, 1), mbar_init(a_ready, 4);
      for (int i = 0; i < NS; ++i) mbar_init(bar_q + i, 1);
      fence_mbar_init();
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // k16 step ks of a 64-query A operand written back by the two column halves: queries [32 hh, 32 hh + 32) sit in the
  // packed columns [32 hh, 32 hh + 16) of the region their S^T / dP^T values came from
  auto a_cols = [](int ks) { return (uint32_t)((ks >> 1) * 32 + (ks & 1) * 8); };

  if (warp == kBTmaWarp) {
    if (lane == 0) {
      mbar_arrive_expect_tx(bar_kv, 2 * TA::BYTES);
      tma_load_tile<DH, 128>(sK, &mk128, &mk32, bar_kv, k0, h, b);
      tma_load_tile<DH, 128>(sV, &mv128, &mv32, bar_kv, k0, h, b);
      const float* lse_bh = prm.lse2 + ((int64_t)b * prm.H + h) * prm.Npad;
      const float* dsc_bh = prm.dsc + ((int64_t)b * prm.H + h) * prm.Npad;
      auto load_stage = [&](int st, int tile) {
        mbar_arrive_expect_tx(bar_q + st, 2 * TB::BYTES + 512);
        tma_load_tile<DH, kBT>(sQ + st * TB::BYTES, &mq128, &mq32, bar_q + st, tile * kBT, h, b);
        tma_load_tile<DH, kBT>(sDO + st * TB::BYTES, &mdo128, &mdo32, bar_q + st, tile * kBT, h, b);
        bulk_g2s(sST + st * 512, lse_bh + tile * kBT, 256, bar_q + st);
        bulk_g2s(sST + st * 512 + 256, dsc_bh + tile * kBT, 256, bar_q + st);
      };
      for (int i = 0; i < NS && i < T_tiles; ++i) load_stage(i, i);
      for (int i = 0; i + NS < T_tiles; ++i) {
        mbar_wait(dkv_done, i & 1);  // Q_i / dO_i (and the statistics of tile i) consumed
        load_stage(i % NS, i + NS);
      }
    }
  } else if (warp == kBMmaWarp) {
    if (lane == 0) {
      auto issue_st = [&](int stage) {
        issue_kmajor<DH, kBM, kBT>(tmem_base, smem_u32(sK), smem_u32(sQ + stage * TB::BYTES));
        if constexpr (X::AT) issue_qk64_ts<DH>(tmem_base + 64, tmem_base + X::KV_VT, smem_u32(sDO + stage * TB::BYTES));
        else issue_kmajor<DH, kBM, kBT>(tmem_base + 64, smem_u32(sV), smem_u32(sDO + stage * TB::BYTES));
      };
      mbar_wait(bar_kv, 0);
      if constexpr (X::AT) mbar_wait(a_ready, 0);
      mbar_wait(bar_q, 0);
      tc_fence_after();
      issue_st(0);
      umma_commit(st_full);
      for (int i = 0; i < T_tiles; ++i) {
        const uint32_t ph = i & 1;
        const int st = i % NS;
        mbar_wait(pt_full, ph);  // P^T_i, dS^T_i in tensor memory (every thread has consumed S^T_i, dP^T_i)
        tc_fence_after();
        issue_ts_mn<DH, kBT>(tmem_base + X::DV_COL, [&](int ks) { return tmem_base + a_cols(ks); },
                             smem_u32(sDO + st * TB::BYTES), i > 0);
        issue_ts_mn<DH, kBT>(tmem_base + X::DK_COL, [&](int ks) { return tmem_base + 64 + a_cols(ks); },
                             smem_u32(sQ + st * TB::BYTES), i > 0);
        umma_commit(dkv_done);
        if (i + 1 < T_tiles) {  // next S^T, dP^T right behind (in-order pipe: P^T_i / dS^T_i are read before the overwrite)
          const int sn = (i + 1) % NS;
          mbar_wait(bar_q + sn, ((i + 1) / NS) & 1);
          tc_fence_after();
          issue_st(sn);
          umma_commit(st_full);
        }
      }
    }
  } else {
    const int rq = warp & 3, hh = warp >> 2;
    const int r = rq * 32 + lane;  // key row of the tile = TMEM lane
    const uint32_t lane_addr = tmem_base + ((uint32_t)(rq * 32) << 16);
    if constexpr (X::AT) {
      if (hh == 0) {  // V rows -> tensor memory, once
        mbar_wait(bar_kv, 0);
        smem_row_to_tmem<X::DHP>(sV, r, lane_addr + X::KV_VT);
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(a_ready);
      }
    }
    const int row = k0 + r;
    const float c = prm.scale_log2e, sc = prm.scale;
    // per-QUERY statistics of the streamed tile: staged in shared memory by the TMA warp (global loads here sat on the
    // critical path of every tile: an L2 round trip after each wake-up); identical addresses for every thread of a warp
    // (broadcast 16-byte loads); the arrays are padded to a multiple of 64 tokens with zeros
    for (int i = 0; i < T_tiles; ++i) {
      const uint32_t ph = i & 1;
      const int st = i % NS;
      const float4* l4 = reinterpret_cast<const float4*>(sST + st * 512) + hh * 8;
      const float4* d4 = l4 + 16;
      mbar_wait(bar_q + st, (i / NS) & 1);  // completed before S^T_i was issued: orders the bulk-copied statistics
      mbar_wait(st_full, ph);
      tc_fence_after();
      uint32_t s[32], dp[32];
      tmem_ld32(lane_addr + hh * 32, s);
      tmem_ld32(lane_addr + 64 + hh * 32, dp);
      tmem_ld_wait();
#pragma unroll
      for (int g = 0; g < 8; ++g) {  // 4 queries per step
        const float4 lq = l4[g], dq4 = d4[g];
        const float p0 = ex2_approx(fmaf(__uint_as_float(s[4 * g + 0]), c, -lq.x));
        const float p1 = ex2_approx(fmaf(__uint_as_float(s[4 * g + 1]), c, -lq.y));
        const float p2 = ex2_approx(fmaf(__uint_as_float(s[4 * g + 2]), c, -lq.z));
        const float p3 = ex2_approx(fmaf(__uint_as_float(s[4 * g + 3]), c, -lq.w));
        const float e0 = p0 * fmaf(__uint_as_float(dp[4 * g + 0]), sc, -dq4.x);
        const float e1 = p1 * fmaf(__uint_as_float(dp[4 * g + 1]), sc, -dq4.y);
        const float e2 = p2 * fmaf(__uint_as_float(dp[4 * g + 2]), sc, -dq4.z);
        const float e3 = p3 * fmaf(__uint_as_float(dp[4 * g + 3]), sc, -dq4.w);
        s[2 * g] = pack_half2(p0, p1), s[2 * g + 1] = pack_half2(p2, p3);
        dp[2 * g] = pack_half2(e0, e1), dp[2 * g + 1] = pack_half2(e2, e3);
      }
      // P^T / dS^T of this thread's 32 queries: fp16 pairs over the first half of the columns its own values came from
      tmem_st16(lane_addr + hh * 32, s);
      tmem_st16(lane_addr + 64 + hh * 32, dp);
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(pt_full);
    }
    mbar_wait(dkv_done, (T_tiles - 1) & 1);
    tc_fence_after();
    const bool rvalid = row < N;
    const int64_t goff = (int64_t)b * prm.g_sb + (int64_t)row * prm.g_sr + h * DH;
    int c0, ncol;
    half_cols<X::DHP>(hh, c0, ncol);
    store_cols_from_tmem<DH>(lane_addr + X::DV_COL, prm.dv + goff, rvalid, c0, ncol);
    store_cols_from_tmem<DH>(lane_addr + X::DK_COL, prm.dk + goff, rvalid, c0, ncol);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kBMmaWarp) {
    __syncwarp();
    tmem_dealloc<X::KV_TCOLS>(tmem_base);
  }
}

template <int DH>
static int launch_spatial_bwd(const void* q, const void* k, const void* v, const void* o, const void* d_o, const float* lse,
                              float* workspace, FABwdParams prm, int64_t q_sb, int64_t q_sr, int64_t k_sb, int64_t k_sr,
                              int64_t v_sb, int64_t v_sr, int64_t o_sb, int64_t o_sr, int64_t do_sb, int64_t do_sr,
                              cudaStream_t st) {
  using X = FABwdCfg<DH>;
  const int B = prm.B, N = prm.N, H = prm.H, Npad = prm.Npad;
  OperandMaps q128, do128, k128, v128, q64, do64, k64, v64;
  int rc = make_operand_maps<DH>(q128, q, H, N, B, q_sr, q_sb, kBM) | make_operand_maps<DH>(do128, d_o, H, N, B, do_sr, do_sb, kBM) |
           make_operand_maps<DH>(k128, k, H, N, B, k_sr, k_sb, kBM) | make_operand_maps<DH>(v128, v, H, N, B, v_sr, v_sb, kBM) |
           make_operand_maps<DH>(q64, q, H, N, B, q_sr, q_sb, kBT) | make_operand_maps<DH>(do64, d_o, H, N, B, do_sr, do_sb, kBT) |
           make_operand_maps<DH>(k64, k, H, N, B, k_sr, k_sb, kBT) | make_operand_maps<DH>(v64, v, H, N, B, v_sr, v_sb, kBT);
  if (rc) {
    return MC_E_CUDA;
  }
  float* lse2 = workspace;
  float* dsc = workspace + (int64_t)B * H * Npad;
  prm.lse2 = lse2, prm.dsc = dsc;
  {
    const int64_t total = (int64_t)B * Npad * H;
    attn_bwd_prep_kernel<DH><<<(unsigned)((total + 255) / 256), 256, 0, st>>>((const __half*)o, (const __half*)d_o, lse, lse2,
                                                                            dsc, o_sb, o_sr, do_sb, do_sr, B, N, Npad, H,
                                                                            prm.scale);
    count_launch();
    if (int e = check_launch("attn_bwd_prep")) return e;
  }
  dim3 grid((N + kBM - 1) / kBM, H, B);
  {
    auto kern = spatial_attn_bwd_dq_kernel<DH>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, X::DQ_SMEM);
    kern<<<grid, kBThreads, X::DQ_SMEM, st>>>(q128.m128, q128.m32, do128.m128, do128.m32, k64.m128, k64.m32, v64.m128, v64.m32, prm);
    count_launch();
    if (int e = check_launch("spatial_attn_bwd_dq")) return e;
  }
  {
    auto kern = spatial_attn_bwd_dkv_kernel<DH>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, X::KV_SMEM);
    kern<<<grid, kBThreads, X::KV_SMEM, st>>>(k128.m128, k128.m32, v128.m128, v128.m32, q64.m128, q64.m32, do64.m128, do64.m32, prm);
    count_launch();
    if (int e = check_launch("spatial_attn_bwd_dkv")) return e;
  }
  return MC_OK;
}

static inline int npad64(int N) { return (N + 63) / 64 * 64; }

}  // namespace mc

extern "C" int64_t mc_spatial_attn_bwd_workspace_bytes(int B, int N, int H) {
  return (int64_t)2 * B * H * mc::npad64(N) * 4;
}

extern "C" int mc_spatial_attn_bwd(const void* q, const void* k, const void* v, const void* o, const void* d_o,
                                   const float* lse, void* dq, void* dk, void* dv, void* workspace, int B, int N, int H,
                                   int DH, int64_t q_stride_b, int64_t q_stride_row, int64_t k_stride_b,
                                   int64_t k_stride_row, int64_t v_stride_b, int64_t v_stride_row, int64_t o_stride_b,
                                   int64_t o_stride_row, int64_t do_stride_b, int64_t do_stride_row, int64_t g_stride_b,
                                   int64_t g_stride_row, float scale, void* stream) {
  using namespace mc;
  const char* entry = "spatial_attn_bwd";
  if (int e = check_attn_operands(entry, {q, k, v, o, d_o, lse, dq, dk, dv, workspace}, {B, N, H})) return e;
  if (int e = check_attn_layout(entry, B, H, {q_stride_b, q_stride_row, k_stride_b, k_stride_row, v_stride_b, v_stride_row,
                                              o_stride_b, o_stride_row, do_stride_b, do_stride_row, g_stride_b, g_stride_row},
                                {q, k, v, o, d_o, dq, dk, dv, workspace}))
    return e;
  FABwdParams prm{};
  prm.dq = (__half*)dq, prm.dk = (__half*)dk, prm.dv = (__half*)dv, prm.g_sb = g_stride_b, prm.g_sr = g_stride_row;
  prm.B = B, prm.N = N, prm.H = H, prm.Npad = npad64(N), prm.scale = scale, prm.scale_log2e = scale * 1.44269504088896340736f;
  cudaStream_t st = (cudaStream_t)stream;
  return dispatch_head_dim(entry, DH, [&](auto dh) {
    return launch_spatial_bwd<decltype(dh)::value>(q, k, v, o, d_o, lse, (float*)workspace, prm, q_stride_b, q_stride_row,
                                                   k_stride_b, k_stride_row, v_stride_b, v_stride_row, o_stride_b,
                                                   o_stride_row, do_stride_b, do_stride_row, st);
  });
}
