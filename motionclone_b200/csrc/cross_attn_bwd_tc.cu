// Text cross-attention backward with respect to Q on tcgen05 tensor cores (TMEM accumulators, tensor-map TMA loads),
// sm_100a. The forward is csrc/cross_attn_fwd_tc.cu; same CTA structure.
//
// The text K / V come from frozen projections of a constant prompt embedding (reference t2v_video_sample.py:67-68;
// utils/motionclone_functions.py:236 differentiates w.r.t. the latents), so dK and dV are never needed on this path:
//   S = Q K^T, dP = dO V^T            two tcgen05.mma chains (M=128 queries, N=80 keys) under one commit
//   P = softmax(scale S)  (exact: the whole key axis is one tile), D = sum_j P_j dP_j
//   dS = scale * P o (dP - D) -> fp16 pairs -> TENSOR MEMORY (over the thread's own S columns)
//   dQ = dS K                          A = dS from tensor memory, B = the SAME shared-memory K tile read MN-major
// One CTA = one (batch, head) and a run of consecutive 128-query tiles; K and V are loaded once per CTA by TMA, the Q and
// dO tiles stream through a two-stage TMA ring; 4 compute warps (thread = query row = TMEM lane) + 1 producer warp.
#include <math.h>

#include "tma_common.cuh"

namespace mc {

constexpr int kXBQ = 128;   // query rows per tile
constexpr int kXBK = 80;    // padded key count
constexpr int kXBThreads = 160;

struct XBParams {
  __half* dq;
  int64_t dq_sb, dq_sr;
  int B, Nq, Nk, H;
  int tiles_per_cta;
  float scale, scale_log2e;
};

template <int DH>
struct XBCfg {
  using TQ = TileParts<DH, kXBQ>;
  using TKV = TileParts<DH, kXBK>;
  static constexpr int DHP = TQ::DHP;
  static constexpr int QS = DH >= 128 ? 1 : 2;  // stages of the (Q, dO) ring
  static constexpr int OFF_Q = 0, OFF_DO = QS * TQ::BYTES, OFF_K = 2 * QS * TQ::BYTES, OFF_V = OFF_K + TKV::BYTES;
  static constexpr int OFF_BAR = OFF_V + TKV::BYTES, SMEM = OFF_BAR + 128 + 1024;
  static constexpr int DP_COL = 80, DQ_COL = 160;  // S / dS at [0,80), dP at [80,160), dQ at [160, 160 + DHP)
  static constexpr int TCOLS = (160 + DHP <= 256) ? 256 : 512;
  static constexpr int CTAS_PER_SM = ctas_per_sm(TCOLS, SMEM);
};

template <int DH>
__global__ void __launch_bounds__(kXBThreads, XBCfg<DH>::CTAS_PER_SM)
cross_attn_bwd_dq_tc_kernel(const __grid_constant__ CUtensorMap mq128, const __grid_constant__ CUtensorMap mq32,
                            const __grid_constant__ CUtensorMap mdo128, const __grid_constant__ CUtensorMap mdo32,
                            const __grid_constant__ CUtensorMap mk128, const __grid_constant__ CUtensorMap mk32,
                            const __grid_constant__ CUtensorMap mv128, const __grid_constant__ CUtensorMap mv32,
                            const XBParams prm) {
  using X = XBCfg<DH>;
  using TQ = typename X::TQ;
  using TKV = typename X::TKV;
  constexpr int DHP = X::DHP, QS = X::QS;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sQ = smem + X::OFF_Q;    // QS stages
  uint8_t* sDO = smem + X::OFF_DO;  // QS stages
  uint8_t* sK = smem + X::OFF_K;
  uint8_t* sV = smem + X::OFF_V;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + X::OFF_BAR);
  uint64_t* bar_kv = bars + 0;     // K, V landed (once)
  uint64_t* q_full = bars + 1;     // [2] Q_i, dO_i landed in stage i % QS
  uint64_t* sdp_full = bars + 3;   // S_i, dP_i in TMEM
  uint64_t* ds_full = bars + 4;    // dS_i in TMEM, S_i / dP_i consumed (4 warp arrivals)
  uint64_t* dq_full = bars + 5;    // dQ_i in TMEM
  uint64_t* dq_free = bars + 6;    // dQ_i copied to registers (4 warp arrivals)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int h = blockIdx.x, b = blockIdx.z;
  const int n_tiles = (prm.Nq + kXBQ - 1) / kXBQ;
  const int t0 = blockIdx.y * prm.tiles_per_cta;
  const int T = min(prm.tiles_per_cta, n_tiles - t0);

  if (warp == 4) {
    tmem_alloc<X::TCOLS>(tmem_slot);
    if (lane == 0) {
      mbar_init(bar_kv, 1), mbar_init(q_full, 1), mbar_init(q_full + 1, 1), mbar_init(sdp_full, 1);
      mbar_init(ds_full, 4), mbar_init(dq_full, 1), mbar_init(dq_free, 4);
      fence_mbar_init();
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 4) {
    if (lane == 0) {
      auto load_q = [&](int i) {
        const int st = i % QS;
        mbar_arrive_expect_tx(q_full + st, 2 * TQ::BYTES);
        tma_load_tile<DH, kXBQ>(sQ + st * TQ::BYTES, &mq128, &mq32, q_full + st, (t0 + i) * kXBQ, h, b);
        tma_load_tile<DH, kXBQ>(sDO + st * TQ::BYTES, &mdo128, &mdo32, q_full + st, (t0 + i) * kXBQ, h, b);
      };
      mbar_arrive_expect_tx(bar_kv, 2 * TKV::BYTES);
      tma_load_tile<DH, kXBK>(sK, &mk128, &mk32, bar_kv, 0, h, b);
      tma_load_tile<DH, kXBK>(sV, &mv128, &mv32, bar_kv, 0, h, b);
      for (int i = 0; i < QS && i < T; ++i) load_q(i);
      mbar_wait(bar_kv, 0);
      mbar_wait(q_full, 0);
      tc_fence_after();
      issue_kmajor<DH, kXBQ, kXBK>(tmem_base, smem_u32(sQ), smem_u32(sK));               // S = Q K^T
      issue_kmajor<DH, kXBQ, kXBK>(tmem_base + X::DP_COL, smem_u32(sDO), smem_u32(sV));  // dP = dO V^T
      umma_commit(sdp_full);
      for (int i = 0; i < T; ++i) {
        const uint32_t ph = i & 1;
        mbar_wait(ds_full, ph);                  // dS_i written; S_i, dP_i consumed (their MMAs - and Q_i / dO_i reads - done)
        if (i > 0) mbar_wait(dq_free, ph ^ 1);   // dQ_{i-1} copied out
        tc_fence_after();
        // dQ = dS K: A = dS in tensor memory, B = K MN-major
        issue_ts_mn<DH, kXBK>(tmem_base + X::DQ_COL, [&](int ks) { return tmem_base + ks * 8; }, smem_u32(sK), false);
        umma_commit(dq_full);
        if (i + QS < T) load_q(i + QS);          // refill the stage of tile i
        if (i + 1 < T) {                         // S_{i+1}, dP_{i+1} right behind dQ_i (in-order pipe)
          const int sn = (i + 1) % QS;
          mbar_wait(q_full + sn, ((i + 1) / QS) & 1);
          tc_fence_after();
          issue_kmajor<DH, kXBQ, kXBK>(tmem_base, smem_u32(sQ + sn * TQ::BYTES), smem_u32(sK));
          issue_kmajor<DH, kXBQ, kXBK>(tmem_base + X::DP_COL, smem_u32(sDO + sn * TQ::BYTES), smem_u32(sV));
          umma_commit(sdp_full);
        }
      }
    }
  } else {
    const uint32_t lane_addr = tmem_base + ((uint32_t)(warp * 32) << 16);
    const float c = prm.scale_log2e, sc = prm.scale;
    const int nk = prm.Nk;
    for (int i = 0; i < T; ++i) {
      const uint32_t ph = i & 1;
      mbar_wait(sdp_full, ph);
      tc_fence_after();
      uint32_t s[kXBK];
      tmem_ld32(lane_addr, s), tmem_ld32(lane_addr + 32, s + 32), tmem_ld16(lane_addr + 64, *reinterpret_cast<uint32_t(*)[16]>(s + 64));
      tmem_ld_wait();
      float mx = -INFINITY;
#pragma unroll
      for (int j = 0; j < kXBK; ++j) {
        if (j >= nk) s[j] = 0xff800000u;
        mx = fmaxf(mx, __uint_as_float(s[j]));
      }
      const float negm = -mx * c;
      float sum = 0.f;
#pragma unroll
      for (int j = 0; j < kXBK; ++j) {
        const float p = ex2_approx(fmaf(__uint_as_float(s[j]), c, negm));
        sum += p;
        s[j] = __float_as_uint(p);
      }
      const float inv = 1.f / sum;
      // P as the forward rounds it (fp16), D = sum_j P_j dP_j, dS = scale * P (dP - D)
      uint32_t dp[kXBK];
      tmem_ld32(lane_addr + X::DP_COL, dp), tmem_ld32(lane_addr + X::DP_COL + 32, dp + 32);
      tmem_ld16(lane_addr + X::DP_COL + 64, *reinterpret_cast<uint32_t(*)[16]>(dp + 64));
      tmem_ld_wait();
      float dsum = 0.f;
#pragma unroll
      for (int j = 0; j < kXBK; ++j) {
        const float p = round_half(__uint_as_float(s[j]) * inv);
        s[j] = __float_as_uint(p);
        dsum = fmaf(p, __uint_as_float(dp[j]), dsum);
      }
#pragma unroll
      for (int j = 0; j < kXBK; j += 2) {
        const float d0 = sc * __uint_as_float(s[j]) * (__uint_as_float(dp[j]) - dsum);
        const float d1 = sc * __uint_as_float(s[j + 1]) * (__uint_as_float(dp[j + 1]) - dsum);
        s[j >> 1] = pack_half2(d0, d1);
      }
      tmem_st32(lane_addr, s);
      tmem_st8(lane_addr + 32, s + 32);
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(ds_full);

      const int row = (t0 + i) * kXBQ + tid;
      __half* orow = prm.dq + (int64_t)b * prm.dq_sb + (int64_t)row * prm.dq_sr + h * DH;
      mbar_wait(dq_full, ph);
      tc_fence_after();
      uint32_t r[DHP];
#pragma unroll
      for (int cc = 0; cc < DHP / 16; ++cc) tmem_ld16(lane_addr + X::DQ_COL + cc * 16, *reinterpret_cast<uint32_t(*)[16]>(r + cc * 16));
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(dq_free);
      if (row < prm.Nq) {
#pragma unroll
        for (int ch = 0; ch < DH / 8; ++ch) {
          uint4 pk;
          pk.x = pack_half2(__uint_as_float(r[ch * 8 + 0]), __uint_as_float(r[ch * 8 + 1]));
          pk.y = pack_half2(__uint_as_float(r[ch * 8 + 2]), __uint_as_float(r[ch * 8 + 3]));
          pk.z = pack_half2(__uint_as_float(r[ch * 8 + 4]), __uint_as_float(r[ch * 8 + 5]));
          pk.w = pack_half2(__uint_as_float(r[ch * 8 + 6]), __uint_as_float(r[ch * 8 + 7]));
          *reinterpret_cast<uint4*>(orow + ch * 8) = pk;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    __syncwarp();
    tmem_dealloc<X::TCOLS>(tmem_base);
  }
}

template <int DH>
static int launch_xattn_bwd(const void* q, const void* k, const void* v, const void* d_o, XBParams prm, int64_t q_sb,
                            int64_t q_sr, int64_t kv_sb, int64_t kv_sr, int64_t do_sb, int64_t do_sr, cudaStream_t st) {
  using X = XBCfg<DH>;
  OperandMaps mq, mdo, mk, mv;
  if (make_operand_maps<DH>(mq, q, prm.H, prm.Nq, prm.B, q_sr, q_sb, kXBQ) ||
      make_operand_maps<DH>(mdo, d_o, prm.H, prm.Nq, prm.B, do_sr, do_sb, kXBQ) ||
      make_operand_maps<DH>(mk, k, prm.H, prm.Nk, prm.B, kv_sr, kv_sb, kXBK) ||
      make_operand_maps<DH>(mv, v, prm.H, prm.Nk, prm.B, kv_sr, kv_sb, kXBK))
    return MC_E_CUDA;
  dim3 grid;
  if (int e = xattn_grid("cross_attn_bwd_dq", (prm.Nq + kXBQ - 1) / kXBQ, prm.H, prm.B, X::CTAS_PER_SM, prm.tiles_per_cta, grid))
    return e;
  auto kern = cross_attn_bwd_dq_tc_kernel<DH>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, X::SMEM);
  kern<<<grid, kXBThreads, X::SMEM, st>>>(mq.m128, mq.m32, mdo.m128, mdo.m32, mk.m128, mk.m32, mv.m128, mv.m32, prm);
  count_launch();
  return check_launch("cross_attn_bwd_dq_tc");
}

}  // namespace mc

extern "C" int mc_cross_attn_bwd_dq(const void* q, const void* k, const void* v, const void* d_o, void* dq, int B, int Nq,
                                    int Nk, int H, int DH, int64_t q_stride_b, int64_t q_stride_row, int64_t kv_stride_b,
                                    int64_t kv_stride_row, int64_t do_stride_b, int64_t do_stride_row,
                                    int64_t dq_stride_b, int64_t dq_stride_row, float scale, void* stream) {
  using namespace mc;
  const char* entry = "cross_attn_bwd_dq";
  if (int e = check_attn_operands(entry, {q, k, v, d_o, dq}, {B, Nq, Nk, H})) return e;
  if (Nk > kXBK) {
    set_error("%s: at most %d keys (text tokens) per tile, got %d", entry, kXBK, Nk);
    return MC_E_UNSUPPORTED;
  }
  if (int e = check_attn_layout(entry, B, H, {q_stride_row, kv_stride_row, dq_stride_row, q_stride_b, kv_stride_b, dq_stride_b,
                                              do_stride_b, do_stride_row}, {q, k, v, d_o, dq}))
    return e;
  XBParams prm{};
  prm.dq = (__half*)dq, prm.dq_sb = dq_stride_b, prm.dq_sr = dq_stride_row;
  prm.B = B, prm.Nq = Nq, prm.Nk = Nk, prm.H = H;
  prm.scale = scale, prm.scale_log2e = scale * 1.44269504088896340736f;
  cudaStream_t st = (cudaStream_t)stream;
  return dispatch_head_dim(entry, DH, [&](auto dh) {
    return launch_xattn_bwd<decltype(dh)::value>(q, k, v, d_o, prm, q_stride_b, q_stride_row, kv_stride_b, kv_stride_row,
                                                 do_stride_b, do_stride_row, st);
  });
}
