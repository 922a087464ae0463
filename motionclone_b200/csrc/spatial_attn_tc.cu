// Spatial self-attention (S1) on 5th-gen tensor cores: tcgen05.mma with TMEM accumulators, operands staged by tensor-map
// TMA (cp.async.bulk.tensor), sm_100a. Forward (this file); the backward (dQ kernel, dK/dV kernel) is csrc/spatial_attn_bwd_tc.cu.
//
// Replaces the xformers seam of `attn1` (reference models/attention.py:190-192, :271-278 -> :535-542,
// xformers.ops.memory_efficient_attention(q, k, v, attn_bias=None)): O = softmax(scale Q K^T) V per (frame, head) over the
// N = h*w tokens of one frame; N = 4096 / 1024 / 256 / 64 and DH = 40 / 80 / 160 / 160 at 16 x 512 x 512. fp32 softmax
// statistics, one rounding of the output (xformers / flash semantics - SURVEY.md appendix "Attention numerics").
//
// Forward, one CTA = one (frame, head, 128-query tile); 192 threads = 4 softmax warps (thread r owns query row r = TMEM
// lane r) + 1 MMA warp (lane 0 issues every tcgen05.mma) + 1 load warp (lane 0 issues every TMA load). Key tiles of 64;
// the score tile S is DOUBLE-BUFFERED in tensor memory so that the tensor pipe computes S_{j+1} while the softmax warps
// are still working on S_j (S_{j+1} = Q K_{j+1}^T does not depend on them):
//   MMA warp:  S_{j+1} = Q K_{j+1}^T   tcgen05.mma M=128 N=64 K=DH, A/B from shared memory -> TMEM buffer (j+1)&1  -> commit s_full[(j+1)&1]
//   softmax :  S_j -> registers (64 fp32 per thread), row max, exp2, P_j -> fp16 pairs -> tcgen05.st back over the first 32
//              columns of the thread's own lane in buffer j&1 (its own, already consumed, S_j)                    -> arrive p_full[j&1]
//   MMA warp:  O += P_j V_j            tcgen05.mma with the A operand (P) read FROM TENSOR MEMORY, B = V_j MN-major straight
//              from its TMA tile (no transpose)                                           -> commit pv_done, stage_free[j % NS]
// Pipe order S0 S1 PV0 S2 PV1 S3 ...: the tensor pipe executes in issue order, so S_{j+2} (which overwrites buffer j&1) is
// behind P V_j (which reads P_j from it). Round-2 ncu of the single-buffered version: the softmax warps spent 35 % of their
// time parked on s_full - S_{j+1} could only be issued behind P V_j, i.e. after the slowest of the four warps had finished
// tile j - and moving half of the exponentials to the FMA pipe changed nothing: the kernel was bound by that serial
// chain, not by MUFU throughput.
// P never touches shared memory: the only shared-memory traffic is TMA writes and the MMA's operand reads. O stays in TMEM
// for the whole key loop; the running maximum is only raised when a row's maximum grows by more than 2^8 (P <= 256 fits
// fp16; exactness is unaffected because numerator and denominator share the reference maximum); only then does the softmax
// warp rescale its 32 rows of O (tcgen05.ld -> multiply -> tcgen05.st). K and V tiles stream through an NS-stage TMA ring.
#include <math.h>

#include "tma_common.cuh"

namespace mc {

constexpr int kFM = 128;         // query rows per CTA (UMMA M)
constexpr int kFBN = 64;         // keys per tile (UMMA N of S, K extent of P V)
constexpr int kFThreads = 192;   // 4 softmax warps + MMA warp + load warp
constexpr int kFMmaWarp = 4, kFTmaWarp = 5;
constexpr float kRescaleThreshold = 8.f;  // log2 units

struct FAParams {
  float* lse;        // [B][H][N] natural-log sum-exp of the scaled scores (nullable)
  __half* o;
  int64_t o_sb, o_sr;
  int B, N, H;
  float scale_log2e;  // scale * log2(e)
};

template <int DH>
struct FACfg {
  using T = TileParts<DH>;            // Q tile (128 rows)
  static constexpr int DHP = T::DHP;
  static constexpr int BN = kFBN;
  using TK = TileParts<DH, BN>;       // K / V tiles
  // Row sums: when the head dim leaves zero-padded columns in the V tile (DH = 40 -> 48), column DH of V is set to 1.0
  // after every TMA load, so accumulator column DH of O = P V IS the row sum (from the same fp16 P as the numerator, at no
  // extra MMA and no extra instruction in the softmax warps). Otherwise the softmax threads add their probabilities.
  static constexpr bool PAD_SUM = DHP > DH && DH < 64;
  static constexpr int NS = DHP <= 80 ? 4 : 3;               // K / V ring depth
  static constexpr int OFF_Q = 0, OFF_K = T::BYTES, OFF_V = OFF_K + NS * TK::BYTES;
  static constexpr int OFF_BAR = OFF_V + NS * TK::BYTES;
  static constexpr int SMEM = OFF_BAR + 256 + 1024;          // + alignment slack (dynamic smem base is 16 B aligned)
  static constexpr int O_COL = 2 * BN;                       // S / P buffers at TMEM [0, BN), [BN, 2 BN); O at [2 BN, 2 BN + DHP)
  static constexpr int ACC_COLS = DHP;
  static constexpr int TCOLS = (O_COL + ACC_COLS <= 256) ? 256 : 512;
  static constexpr int CTAS_PER_SM = ctas_per_sm(TCOLS, SMEM);
};

// all lanes of the load warp: element DH of every key row of a landed V tile := 1.0 (see FACfg::PAD_SUM)
template <int DH>
__device__ __forceinline__ void write_v_ones(uint8_t* sVstage, int lane) {
  using X = FACfg<DH>;
  constexpr int ch = DH / 8;  // the 16-byte chunk holding elements [DH, DH + 8): zero-filled by the TMA unit
  for (int r = lane; r < X::BN; r += 32)
    *reinterpret_cast<uint4*>(sVstage + sw128_chunk_off(r, ch)) = make_uint4(0x00003C00u, 0u, 0u, 0u);
  fence_proxy_async();
  __syncwarp();
}

template <int DH>
__global__ void __launch_bounds__(kFThreads, FACfg<DH>::CTAS_PER_SM)
spatial_attn_fwd_kernel(const __grid_constant__ CUtensorMap mq128, const __grid_constant__ CUtensorMap mk128,
                        const __grid_constant__ CUtensorMap mv128, const __grid_constant__ CUtensorMap mq32,
                        const __grid_constant__ CUtensorMap mk32, const __grid_constant__ CUtensorMap mv32,
                        const FAParams prm) {
  using X = FACfg<DH>;
  using T = TileParts<DH>;
  using TK = typename X::TK;
  constexpr int DHP = X::DHP, BN = X::BN, NS = X::NS;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sQ = smem + X::OFF_Q;
  uint8_t* sK = smem + X::OFF_K;   // NS stages
  uint8_t* sV = smem + X::OFF_V;   // NS stages
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + X::OFF_BAR);
  uint64_t* bar_q = bars + 0;        // Q landed                                         (tx)
  uint64_t* s_full = bars + 1;       // [2] S_j in TMEM buffer j & 1                      (tcgen05.commit)
  uint64_t* p_full = bars + 3;       // [2] P_j in TMEM buffer j & 1, S_j consumed        (4 warp arrivals)
  uint64_t* pv_done = bars + 5;      // O += P_j V_j completed                            (tcgen05.commit)
  uint64_t* kv_full = bars + 6;      // [NS] K_j and V_j landed in stage j % NS            (tx)
  uint64_t* v_ready = bars + 10;     // [NS] ones column written into V_j (PAD_SUM)        (1 arrival)
  uint64_t* stage_free = bars + 14;  // [NS] S_j and P V_j completed: stage j % NS may be refilled (tcgen05.commit)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 18);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int qt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int q0 = qt * kFM, N = prm.N;
  const int T_tiles = (N + BN - 1) / BN;

  if (warp == kFMmaWarp) {
    tmem_alloc<X::TCOLS>(tmem_slot);
    if (lane == 0) {
      mbar_init(bar_q, 1), mbar_init(pv_done, 1);
      for (int i = 0; i < 2; ++i) mbar_init(s_full + i, 1), mbar_init(p_full + i, 4);
      for (int i = 0; i < NS; ++i) mbar_init(kv_full + i, 1), mbar_init(v_ready + i, 1), mbar_init(stage_free + i, 1);
      fence_mbar_init();
      tma_prefetch_desc(&mq128), tma_prefetch_desc(&mk128), tma_prefetch_desc(&mv128);
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == kFTmaWarp) {
    // ================= load warp: lane 0 issues every TMA load; all lanes write the ones column =================
    auto load_kv = [&](int j) {
      const int st = j % NS;
      mbar_arrive_expect_tx(kv_full + st, 2 * TK::BYTES);
      tma_load_tile<DH, BN>(sK + st * TK::BYTES, &mk128, &mk32, kv_full + st, j * BN, h, b);
      tma_load_tile<DH, BN>(sV + st * TK::BYTES, &mv128, &mv32, kv_full + st, j * BN, h, b);
    };
    if (lane == 0) {
      mbar_arrive_expect_tx(bar_q, T::BYTES);
      tma_load_tile<DH>(sQ, &mq128, &mq32, bar_q, q0, h, b);
      for (int j = 0; j < NS && j < T_tiles; ++j) load_kv(j);
    }
    for (int j = 0; j < T_tiles; ++j) {
      if constexpr (X::PAD_SUM) {
        const int st = j % NS;
        mbar_wait(kv_full + st, (j / NS) & 1);
        write_v_ones<DH>(sV + st * TK::BYTES, lane);
        if (lane == 0) mbar_arrive(v_ready + st);
      }
      if (j >= 1 && j - 1 + NS < T_tiles) {  // refill the stage of tile j - 1 once its MMAs have completed
        mbar_wait(stage_free + (j - 1) % NS, ((j - 1) / NS) & 1);
        if (lane == 0) load_kv(j - 1 + NS);
      }
      __syncwarp();
    }
  } else if (warp == kFMmaWarp) {
    // ================= MMA warp: lane 0 issues every MMA =================
    if (lane == 0) {
      mbar_wait(bar_q, 0);
      mbar_wait(kv_full, 0);
      tc_fence_after();
      issue_kmajor<DH, kFM, BN>(tmem_base, smem_u32(sQ), smem_u32(sK));
      umma_commit(s_full);
      for (int j = 0; j < T_tiles; ++j) {
        const int st = j % NS, buf = j & 1;
        if (j + 1 < T_tiles) {  // S_{j+1} into the other buffer while the softmax warps work on S_j
          const int sn = (j + 1) % NS;
          mbar_wait(kv_full + sn, ((j + 1) / NS) & 1);
          tc_fence_after();
          issue_kmajor<DH, kFM, BN>(tmem_base + (buf ^ 1) * BN, smem_u32(sQ), smem_u32(sK + sn * TK::BYTES));
          umma_commit(s_full + (buf ^ 1));
        }
        mbar_wait(p_full + buf, (j >> 1) & 1);  // every softmax thread has consumed S_j and written P_j
        if constexpr (X::PAD_SUM) mbar_wait(v_ready + st, (j / NS) & 1);
        tc_fence_after();
        issue_ts_mn<DH, BN>(tmem_base + X::O_COL, [p = tmem_base + buf * BN](int ks) { return p + ks * 8; },
                            smem_u32(sV + st * TK::BYTES), j > 0);
        umma_commit(pv_done);
        umma_commit(stage_free + st);
      }
    }
  } else {
    // ================= softmax warps: thread = query row =================
    const uint32_t lane_addr = tmem_base + ((uint32_t)(warp * 32) << 16);
    const float c = prm.scale_log2e;
    float m_used = -INFINITY, l_thr = 0.f;  // l_thr: thread-side row sum (unused when the V pad column carries it)
    for (int j = 0; j < T_tiles; ++j) {
      const uint32_t ph = j & 1;
      const uint32_t sbuf = lane_addr + (j & 1) * BN;
      mbar_wait(s_full + (j & 1), (j >> 1) & 1);
      tc_fence_after();
      uint32_t s[BN];
#pragma unroll
      for (int cc = 0; cc < BN / 32; ++cc) tmem_ld32(sbuf + cc * 32, s + cc * 32);
      tmem_ld_wait();

      const int kvalid = N - j * BN;  // keys of this tile that exist (>= 1)
      if (kvalid < BN) {
#pragma unroll
        for (int i = 0; i < BN; ++i)
          if (i >= kvalid) s[i] = 0xff800000u;  // -inf
      }
      float mx0 = __uint_as_float(s[0]), mx1 = __uint_as_float(s[1]), mx2 = __uint_as_float(s[2]),
            mx3 = __uint_as_float(s[3]);
#pragma unroll
      for (int i = 4; i < BN; i += 4) {
        mx0 = fmaxf(mx0, __uint_as_float(s[i])), mx1 = fmaxf(mx1, __uint_as_float(s[i + 1]));
        mx2 = fmaxf(mx2, __uint_as_float(s[i + 2])), mx3 = fmaxf(mx3, __uint_as_float(s[i + 3]));
      }
      const float mxc = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3)) * c;
      if (j == 0) {
        m_used = mxc;
      } else {
        const bool grow = mxc - m_used > kRescaleThreshold;
        if (__any_sync(0xffffffffu, grow)) {
          const float m_new = grow ? mxc : m_used;
          const float alpha = ex2_approx(m_used - m_new);
          m_used = m_new;
          l_thr *= alpha;
          mbar_wait(pv_done, ph ^ 1);  // O holds tiles 0..j-1 (P V_j cannot start before this warp's p_full arrival)
          tc_fence_after();
#pragma unroll
          for (int cc = 0; cc < X::ACC_COLS / 16; ++cc) {
            uint32_t r[16];
            tmem_ld16(lane_addr + X::O_COL + cc * 16, r);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) * alpha);
            tmem_st16(lane_addr + X::O_COL + cc * 16, r);
          }
        }
      }
      // p = exp2(s*c - m_used), packed to fp16 pairs in place (s[0 .. BN/2) then hold the BN probabilities)
      const float negm = -m_used;
      float l0 = 0.f, l1 = 0.f;
#pragma unroll
      for (int i = 0; i < BN; i += 2) {
        float p0, p1;
        ex2_pair(i >> 1, __uint_as_float(s[i]), __uint_as_float(s[i + 1]), c, negm, p0, p1);
        if constexpr (!X::PAD_SUM) l0 += p0, l1 += p1;
        s[i >> 1] = pack_half2(p0, p1);
      }
      if constexpr (!X::PAD_SUM) l_thr += l0 + l1;
      tmem_st32(sbuf, s);  // P over the consumed S (first BN / 2 columns of the buffer)
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_full + (j & 1));
    }
    // ---- epilogue: O / l -> fp16 -> global; log-sum-exp for the backward ----
    // S_{T-1} was issued BEFORE P V_{T-2}, so having consumed it only proves P V_{T-3} complete: a single parity wait for
    // phase T-1 could be satisfied by the still-incomplete phase T-2 looking like "phase T-3 done". Wait for both in order.
    if (T_tiles >= 2) mbar_wait(pv_done, (T_tiles - 2) & 1);
    mbar_wait(pv_done, (T_tiles - 1) & 1);
    tc_fence_after();
    const int row = q0 + tid;
    float l = l_thr;
    if constexpr (X::PAD_SUM) {  // accumulator column DH = sum_j P_j * 1
      uint32_t r[16];
      tmem_ld16(lane_addr + X::O_COL + (DH / 16) * 16, r);
      tmem_ld_wait();
      l = __uint_as_float(r[DH % 16]);
    }
    const float inv = 1.f / l;
    __half* orow = prm.o + (int64_t)b * prm.o_sb + (int64_t)row * prm.o_sr + h * DH;
#pragma unroll
    for (int cc = 0; cc < DHP / 16; ++cc) {
      uint32_t r[16];
      tmem_ld16(lane_addr + X::O_COL + cc * 16, r);
      tmem_ld_wait();
      if (row < N) {
#pragma unroll
        for (int half8 = 0; half8 < 2; ++half8) {
          if (cc * 16 + half8 * 8 < DH) {
            uint4 pk;
            pk.x = pack_half2(__uint_as_float(r[half8 * 8 + 0]) * inv, __uint_as_float(r[half8 * 8 + 1]) * inv);
            pk.y = pack_half2(__uint_as_float(r[half8 * 8 + 2]) * inv, __uint_as_float(r[half8 * 8 + 3]) * inv);
            pk.z = pack_half2(__uint_as_float(r[half8 * 8 + 4]) * inv, __uint_as_float(r[half8 * 8 + 5]) * inv);
            pk.w = pack_half2(__uint_as_float(r[half8 * 8 + 6]) * inv, __uint_as_float(r[half8 * 8 + 7]) * inv);
            *reinterpret_cast<uint4*>(orow + cc * 16 + half8 * 8) = pk;
          }
        }
      }
    }
    if (prm.lse != nullptr && row < N)
      prm.lse[((int64_t)b * prm.H + h) * N + row] = (m_used + log2f(l)) * 0.6931471805599453f;
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kFMmaWarp) {
    __syncwarp();
    tmem_dealloc<X::TCOLS>(tmem_base);
  }
}

template <int DH>
static int launch_spatial_fwd(const void* q, const void* k, const void* v, const FAParams& prm, int64_t q_sb, int64_t q_sr,
                              int64_t k_sb, int64_t k_sr, int64_t v_sb, int64_t v_sr, cudaStream_t st) {
  using X = FACfg<DH>;
  OperandMaps mq, mk, mv;
  if (make_operand_maps<DH>(mq, q, prm.H, prm.N, prm.B, q_sr, q_sb, kFM) ||
      make_operand_maps<DH>(mk, k, prm.H, prm.N, prm.B, k_sr, k_sb, X::BN) ||
      make_operand_maps<DH>(mv, v, prm.H, prm.N, prm.B, v_sr, v_sb, X::BN)) {
    return MC_E_CUDA;
  }
  auto kern = spatial_attn_fwd_kernel<DH>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, X::SMEM);
  dim3 grid((prm.N + kFM - 1) / kFM, prm.H, prm.B);
  kern<<<grid, kFThreads, X::SMEM, st>>>(mq.m128, mk.m128, mv.m128, mq.m32, mk.m32, mv.m32, prm);
  count_launch();
  return check_launch("spatial_attn_fwd");
}

}  // namespace mc

extern "C" int mc_spatial_attn_fwd(const void* q, const void* k, const void* v, void* o, float* lse, int B, int N, int H,
                                   int DH, int64_t q_stride_b, int64_t q_stride_row, int64_t k_stride_b,
                                   int64_t k_stride_row, int64_t v_stride_b, int64_t v_stride_row, int64_t o_stride_b,
                                   int64_t o_stride_row, float scale, void* stream) {
  using namespace mc;
  const char* entry = "spatial_attn_fwd";
  if (int e = check_attn_operands(entry, {q, k, v, o}, {B, N, H})) return e;
  if (int e = check_attn_layout(entry, B, H, {q_stride_b, q_stride_row, k_stride_b, k_stride_row, v_stride_b, v_stride_row,
                                              o_stride_b, o_stride_row}, {q, k, v, o}))
    return e;
  FAParams prm{};
  prm.lse = lse, prm.o = (__half*)o, prm.o_sb = o_stride_b, prm.o_sr = o_stride_row;
  prm.B = B, prm.N = N, prm.H = H;
  prm.scale_log2e = scale * 1.44269504088896340736f;
  cudaStream_t st = (cudaStream_t)stream;
  return dispatch_head_dim(entry, DH, [&](auto dh) {
    return launch_spatial_fwd<decltype(dh)::value>(q, k, v, prm, q_stride_b, q_stride_row, k_stride_b, k_stride_row,
                                                   v_stride_b, v_stride_row, st);
  });
}
