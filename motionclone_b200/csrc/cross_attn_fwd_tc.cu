// Text cross-attention forward on 5th-gen tensor cores (tcgen05) with TMEM accumulators and tensor-map TMA loads, sm_100a.
//
// Replaces the xformers seam for `attn2` (reference models/attention.py:193-201, :280-285 -> :535-542,
// xformers.ops.memory_efficient_attention): O = softmax(scale * Q K^T) V with Q [b, f*N, C] (all frames of one prompt:
// the text K/V [b, 77, C] are shared by every frame) and 8 heads of DH in {40, 80, 160}. The op is HBM-bound (Q read +
// O written, 4 flop/B): what matters is bytes in flight and nothing else.
//
// One CTA = one (batch, head) and a run of consecutive 128-query tiles; 160 threads = 4 softmax warps (thread r = query
// row r = TMEM lane r) + 1 producer warp whose lane 0 issues every TMA load and MMA. K and V (77 -> 80 rows) are loaded
// ONCE per CTA; Q tiles stream through a two-stage TMA ring. The whole key axis is one tile, so the softmax is exact in
// one pass (no online rescaling). Per query tile i:
//   producer:  S = Q_i K^T        tcgen05.mma M=128 N=80 K=DH, operands from shared memory (SW128 / SW32 parts)
//   softmax :  S -> registers, row max, exp2, row sum, P -> fp16 pairs -> tcgen05.st over its own S columns
//   producer:  O = P V            tcgen05.mma with A = P from TENSOR MEMORY, B = V MN-major from its TMA tile; then S_{i+1}
//   softmax :  O -> registers, / row sum -> fp16 -> global (each thread its row's DH contiguous values)
// Four CTAs share an SM at DH = 40 (TMEM 128 columns, 52 KB shared memory each), so loads, exponentials, MMAs and stores
// of different tiles overlap across CTAs as well as across the two Q stages.
#include <math.h>

#include "tma_common.cuh"

namespace mc {

constexpr int kXQ = 128;        // query rows per tile (UMMA M)
constexpr int kXK = 80;         // padded key count (UMMA N of S, K extent of P V); 77 text tokens
constexpr int kXFThreads = 160;

struct XFParams {
  __half* o;
  int64_t o_sb, o_sr;
  int B, Nq, Nk, H;
  int tiles_per_cta;
  float scale_log2e;
};

template <int DH>
struct XFCfg {
  using TQ = TileParts<DH, kXQ>;
  using TKV = TileParts<DH, kXK>;
  static constexpr int DHP = TQ::DHP;
  static constexpr int QS = DH >= 128 ? 1 : 2;  // Q stages
  static constexpr int OFF_Q = 0, OFF_K = QS * TQ::BYTES, OFF_V = OFF_K + TKV::BYTES, OFF_BAR = OFF_V + TKV::BYTES;
  static constexpr int SMEM = OFF_BAR + 128 + 1024;
  static constexpr int O_COL = kXK;  // S / P at TMEM [0, 80), O at [80, 80 + DHP)
  static constexpr int TCOLS = (kXK + DHP <= 128) ? 128 : 256;
  static constexpr int CTAS_PER_SM = ctas_per_sm(TCOLS, SMEM);
};

template <int DH>
__global__ void __launch_bounds__(kXFThreads, XFCfg<DH>::CTAS_PER_SM)
cross_attn_fwd_tc_kernel(const __grid_constant__ CUtensorMap mq128, const __grid_constant__ CUtensorMap mq32,
                         const __grid_constant__ CUtensorMap mk128, const __grid_constant__ CUtensorMap mk32,
                         const __grid_constant__ CUtensorMap mv128, const __grid_constant__ CUtensorMap mv32,
                         const XFParams prm) {
  using X = XFCfg<DH>;
  using TQ = typename X::TQ;
  using TKV = typename X::TKV;
  constexpr int DHP = X::DHP, QS = X::QS;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sQ = smem + X::OFF_Q;   // QS stages
  uint8_t* sK = smem + X::OFF_K;
  uint8_t* sV = smem + X::OFF_V;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + X::OFF_BAR);
  uint64_t* bar_kv = bars + 0;     // K, V landed (once)
  uint64_t* q_full = bars + 1;     // [2] Q_i landed in stage i % QS
  uint64_t* s_full = bars + 3;     // S_i in TMEM
  uint64_t* p_full = bars + 4;     // P_i in TMEM, S_i consumed (4 warp arrivals)
  uint64_t* o_full = bars + 5;     // O_i = P_i V in TMEM
  uint64_t* o_free = bars + 6;     // O_i copied to registers (4 warp arrivals)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int h = blockIdx.x, b = blockIdx.z;  // heads fastest: the 8 CTAs sharing Q / O rows run together
  const int n_tiles = (prm.Nq + kXQ - 1) / kXQ;
  const int t0 = blockIdx.y * prm.tiles_per_cta;
  const int T = min(prm.tiles_per_cta, n_tiles - t0);

  if (warp == 4) {
    tmem_alloc<X::TCOLS>(tmem_slot);
    if (lane == 0) {
      mbar_init(bar_kv, 1), mbar_init(q_full, 1), mbar_init(q_full + 1, 1), mbar_init(s_full, 1);
      mbar_init(p_full, 4), mbar_init(o_full, 1), mbar_init(o_free, 4);
      fence_mbar_init();
      tma_prefetch_desc(&mq128), tma_prefetch_desc(&mk128), tma_prefetch_desc(&mv128);
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 4) {
    if (lane == 0) {
      auto issue_s = [&](int stage) {  // S = Q K^T
        issue_kmajor<DH, kXQ, kXK>(tmem_base, smem_u32(sQ + stage * TQ::BYTES), smem_u32(sK));
      };
      mbar_arrive_expect_tx(bar_kv, 2 * TKV::BYTES);
      tma_load_tile<DH, kXK>(sK, &mk128, &mk32, bar_kv, 0, h, b);
      tma_load_tile<DH, kXK>(sV, &mv128, &mv32, bar_kv, 0, h, b);
      for (int i = 0; i < QS && i < T; ++i) {
        mbar_arrive_expect_tx(q_full + i, TQ::BYTES);
        tma_load_tile<DH, kXQ>(sQ + i * TQ::BYTES, &mq128, &mq32, q_full + i, (t0 + i) * kXQ, h, b);
      }
      mbar_wait(bar_kv, 0);
      mbar_wait(q_full, 0);
      tc_fence_after();
      issue_s(0);
      umma_commit(s_full);
      for (int i = 0; i < T; ++i) {
        const uint32_t ph = i & 1;
        mbar_wait(p_full, ph);                     // P_i written, S_i consumed (so S_i's MMA - and Q_i's reads - are done)
        if (i > 0) mbar_wait(o_free, ph ^ 1);      // O_{i-1} copied out
        tc_fence_after();
        // O = P V: A = P in tensor memory, B = V MN-major
        issue_ts_mn<DH, kXK>(tmem_base + X::O_COL, [&](int ks) { return tmem_base + ks * 8; }, smem_u32(sV), false);
        umma_commit(o_full);
        if (i + QS < T) {                          // refill Q_i's stage with tile i + QS
          const int st = i % QS;
          mbar_arrive_expect_tx(q_full + st, TQ::BYTES);
          tma_load_tile<DH, kXQ>(sQ + st * TQ::BYTES, &mq128, &mq32, q_full + st, (t0 + i + QS) * kXQ, h, b);
        }
        if (i + 1 < T) {                           // S_{i+1} right behind P V_i (in-order pipe)
          const int sn = (i + 1) % QS;
          mbar_wait(q_full + sn, ((i + 1) / QS) & 1);
          tc_fence_after();
          issue_s(sn);
          umma_commit(s_full);
        }
      }
    }
  } else {
    const uint32_t lane_addr = tmem_base + ((uint32_t)(warp * 32) << 16);
    const float c = prm.scale_log2e;
    const int nk = prm.Nk;
    for (int i = 0; i < T; ++i) {
      const uint32_t ph = i & 1;
      mbar_wait(s_full, ph);
      tc_fence_after();
      uint32_t s[kXK];
      tmem_ld32(lane_addr, s), tmem_ld32(lane_addr + 32, s + 32), tmem_ld16(lane_addr + 64, *reinterpret_cast<uint32_t(*)[16]>(s + 64));
      tmem_ld_wait();
      float mx = -INFINITY;
#pragma unroll
      for (int j = 0; j < kXK; ++j) {
        if (j >= nk) s[j] = 0xff800000u;  // keys past the end: -inf
        mx = fmaxf(mx, __uint_as_float(s[j]));
      }
      const float negm = -mx * c;
      float sum0 = 0.f, sum1 = 0.f;
#pragma unroll
      for (int j = 0; j < kXK; j += 2) {
        const float p0 = ex2_approx(fmaf(__uint_as_float(s[j]), c, negm));
        const float p1 = ex2_approx(fmaf(__uint_as_float(s[j + 1]), c, negm));
        sum0 += p0, sum1 += p1;
        s[j >> 1] = pack_half2(p0, p1);
      }
      tmem_st32(lane_addr, s);
      tmem_st8(lane_addr + 32, s + 32);
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_full);

      const float inv = 1.f / (sum0 + sum1);
      const int row = (t0 + i) * kXQ + tid;
      __half* orow = prm.o + (int64_t)b * prm.o_sb + (int64_t)row * prm.o_sr + h * DH;
      mbar_wait(o_full, ph);
      tc_fence_after();
      uint32_t r[DHP];
#pragma unroll
      for (int cc = 0; cc < DHP / 16; ++cc) tmem_ld16(lane_addr + X::O_COL + cc * 16, *reinterpret_cast<uint32_t(*)[16]>(r + cc * 16));
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(o_free);
      if (row < prm.Nq) {
#pragma unroll
        for (int ch = 0; ch < DH / 8; ++ch) {
          uint4 pk;
          pk.x = pack_half2(__uint_as_float(r[ch * 8 + 0]) * inv, __uint_as_float(r[ch * 8 + 1]) * inv);
          pk.y = pack_half2(__uint_as_float(r[ch * 8 + 2]) * inv, __uint_as_float(r[ch * 8 + 3]) * inv);
          pk.z = pack_half2(__uint_as_float(r[ch * 8 + 4]) * inv, __uint_as_float(r[ch * 8 + 5]) * inv);
          pk.w = pack_half2(__uint_as_float(r[ch * 8 + 6]) * inv, __uint_as_float(r[ch * 8 + 7]) * inv);
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
static int launch_xattn_fwd(const void* q, const void* k, const void* v, XFParams prm, int64_t q_sb, int64_t q_sr, int64_t kv_sb,
                            int64_t kv_sr, cudaStream_t st) {
  using X = XFCfg<DH>;
  OperandMaps mq, mk, mv;
  if (make_operand_maps<DH>(mq, q, prm.H, prm.Nq, prm.B, q_sr, q_sb, kXQ) ||
      make_operand_maps<DH>(mk, k, prm.H, prm.Nk, prm.B, kv_sr, kv_sb, kXK) ||
      make_operand_maps<DH>(mv, v, prm.H, prm.Nk, prm.B, kv_sr, kv_sb, kXK))
    return MC_E_CUDA;
  dim3 grid;
  if (int e = xattn_grid("cross_attn_fwd", (prm.Nq + kXQ - 1) / kXQ, prm.H, prm.B, X::CTAS_PER_SM, prm.tiles_per_cta, grid))
    return e;
  auto kern = cross_attn_fwd_tc_kernel<DH>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, X::SMEM);
  kern<<<grid, kXFThreads, X::SMEM, st>>>(mq.m128, mq.m32, mk.m128, mk.m32, mv.m128, mv.m32, prm);
  count_launch();
  return check_launch("cross_attn_fwd_tc");
}

}  // namespace mc

extern "C" int mc_cross_attn_fwd(const void* q, const void* k, const void* v, void* o, int B, int Nq, int Nk, int H, int DH,
                                 int64_t q_stride_b, int64_t q_stride_row, int64_t kv_stride_b, int64_t kv_stride_row,
                                 int64_t o_stride_b, int64_t o_stride_row, float scale, void* stream) {
  using namespace mc;
  const char* entry = "cross_attn_fwd";
  if (int e = check_attn_operands(entry, {q, k, v, o}, {B, Nq, Nk, H})) return e;
  if (Nk > kXK) {
    set_error("%s: at most %d keys (text tokens) per tile, got %d", entry, kXK, Nk);
    return MC_E_UNSUPPORTED;
  }
  if (int e = check_attn_layout(entry, B, H, {q_stride_row, kv_stride_row, o_stride_row, q_stride_b, kv_stride_b, o_stride_b},
                                {q, k, v, o}))
    return e;
  XFParams prm{};
  prm.o = (__half*)o, prm.o_sb = o_stride_b, prm.o_sr = o_stride_row;
  prm.B = B, prm.Nq = Nq, prm.Nk = Nk, prm.H = H;
  prm.scale_log2e = scale * 1.44269504088896340736f;
  cudaStream_t st = (cudaStream_t)stream;
  return dispatch_head_dim(entry, DH, [&](auto dh) {
    return launch_xattn_fwd<decltype(dh)::value>(q, k, v, prm, q_stride_b, q_stride_row, kv_stride_b, kv_stride_row, st);
  });
}
