// The tcgen05 attention layer (sm_100a): TMA tensor maps (cp.async.bulk.tensor, SASS UTMALDG), swizzled UMMA
// shared-memory descriptors, MMA issue, TMEM loads / stores, and the host-side pieces every attention entry point shares
// (operand maps, head-dim dispatch, argument checks).
//
// An attention operand tile is [128 rows][DH] fp16 (rows = tokens of one frame / head, DH contiguous in global memory).
// In shared memory it is a sequence of PARTS along DH, each landed by ONE tensor-map load:
//   SW128 part: [128 rows][64 elements = 128 B], CU_TENSOR_MAP_SWIZZLE_128B   (16 KB; 1024-byte aligned)
//   SW32  part: [128 rows][16 elements =  32 B], CU_TENSOR_MAP_SWIZZLE_32B    ( 4 KB)
// DH = 40 -> one SW128 part whose columns 40..63 are zero-filled by the TMA unit (the map's innermost extent is DH, the
// box is 64 wide: out-of-bounds elements read as 0); DH = 80 -> SW128 + SW32; DH = 160 -> 2 x SW128 + 2 x SW32.
// The same bytes serve as
//   K-major operand  (rows = M or N, DH = K):  canonical  Swizzle<3,4,3> o ((8,n),2):((8,SBO),1)   [units of 16 B]
//   MN-major operand (DH = M or N, rows = K):  canonical  Swizzle<3,4,3> o ((8,n),(8,k)):((1,LBO),(8,SBO))
// so V needs no transpose for P V, and K / Q / dO tiles are shared between the GEMMs of the backward pass.
#pragma once
#include <cuda.h>

#include <initializer_list>
#include <type_traits>

#include "mc_common.cuh"

namespace mc {

// ---- operand-tile geometry ----
template <int DH, int ROWS = 128>
struct TileParts {
  static_assert(DH % 8 == 0, "head dim must be a multiple of 8 (16-byte rows)");
  static_assert(ROWS % 8 == 0 && ROWS <= 256, "tile rows");
  static constexpr int N64 = DH >= 64 ? DH / 64 : 1;   // SW128 parts
  static constexpr int REM = DH >= 64 ? DH % 64 : 0;
  static_assert(REM % 16 == 0, "head dims above 64 must be 64*a + 16*b");
  static constexpr int N16 = REM / 16;                 // SW32 parts
  static constexpr int DHP = DH >= 64 ? DH : (DH + 15) / 16 * 16;  // extent seen by the MMA (zero-padded below 64)
  static constexpr int KS64 = DH >= 64 ? 4 : DHP / 16;             // k16 steps per SW128 part when DH is the K dim
  static constexpr int W64 = DH >= 64 ? 64 : DHP;                  // N extent per SW128 part when DH is the N dim
  static constexpr int P64 = ROWS * 128, P16 = ROWS * 32;          // bytes per part
  static constexpr int BYTES = N64 * P64 + N16 * P16;
  static constexpr int KSTEPS = N64 * KS64 + N16;
  __host__ __device__ static constexpr int part64_off(int p) { return p * P64; }
  __host__ __device__ static constexpr int part16_off(int p) { return N64 * P64 + p * P16; }
};

// CTAs of one kernel resident on an SM: bounded by tensor memory (512 columns) and by shared memory (227 KB)
__host__ __device__ constexpr int ctas_per_sm(int tmem_cols, int smem_bytes) {
  const int by_tmem = 512 / tmem_cols, by_smem = (227 * 1024) / smem_bytes;
  return by_tmem < by_smem ? by_tmem : (by_smem < 1 ? 1 : by_smem);
}

// ---- host: tensor-map encode through the runtime's driver entry point (no link-time dependency on libcuda) ----
typedef CUresult (*mc_encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                       const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                       CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline mc_encode_tiled_fn tensor_map_encoder() {
  static mc_encode_tiled_fn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return (mc_encode_tiled_fn)p;
  }();
  return fn;
}

// fp16 tensor [frames][rows][heads][DH]: element (b, r, h, e) at base + b*stride_b + r*stride_r + h*DH + e (elements).
// Box = (box_e, 1 head, 128 rows, 1 frame); coordinates (e0, h, r0, b). Returns 0 on success.
inline int make_attn_tensor_map(CUtensorMap* map, const void* base, int DH, int H, int64_t rows, int64_t frames,
                                int64_t stride_r, int64_t stride_b, int box_e, int box_rows, bool swizzle128) {
  mc_encode_tiled_fn enc = tensor_map_encoder();
  // The encoder is a DRIVER entry point: it needs the primary context current on the calling thread. A thread that has
  // not yet made a runtime call (autograd's backward worker on its first node) has none -> CUDA_ERROR_INVALID_CONTEXT.
  static thread_local bool ctx_bound = false;
  if (!ctx_bound) {
    cudaFree(nullptr);  // binds the runtime's primary context to this thread (no-op otherwise)
    ctx_bound = true;
  }
  if (!enc) {
    set_error("cuTensorMapEncodeTiled: driver entry point unavailable (cudaGetDriverEntryPoint failed)");
    return -1;
  }
  cuuint64_t gdim[4] = {(cuuint64_t)DH, (cuuint64_t)H, (cuuint64_t)rows, (cuuint64_t)frames};
  cuuint64_t gstr[3] = {(cuuint64_t)DH * 2, (cuuint64_t)stride_r * 2, (cuuint64_t)stride_b * 2};
  if (frames == 1) gstr[2] = gstr[1] * (cuuint64_t)rows;  // unused dimension: any legal stride
  cuuint32_t box[4] = {(cuuint32_t)box_e, 1u, (cuuint32_t)box_rows, 1u};
  cuuint32_t estr[4] = {1u, 1u, 1u, 1u};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(base), gdim, gstr, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_32B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    set_error("cuTensorMapEncodeTiled -> CUresult %d: base %p dims (%d, %d, %lld, %lld) strides (%lld, %lld) elements, box "
              "(%d, 1, %d, 1), swizzle %s", (int)r, base, DH, H, (long long)rows, (long long)frames, (long long)stride_r,
              (long long)stride_b, box_e, box_rows, swizzle128 ? "128B" : "32B");
  return r == CUDA_SUCCESS ? 0 : (int)r;
}

// the two maps of one operand tensor (box height `box_rows`): SW128 parts and SW32 parts; the SW32 map is only encoded
// when the head dim has 16-wide parts
struct OperandMaps {
  CUtensorMap m128, m32;
};
template <int DH>
inline int make_operand_maps(OperandMaps& m, const void* base, int H, int rows, int frames, int64_t stride_r,
                             int64_t stride_b, int box_rows) {
  int rc = make_attn_tensor_map(&m.m128, base, DH, H, rows, frames, stride_r, stride_b, 64, box_rows, true);
  if (rc) return rc;
  if (TileParts<DH>::N16 > 0) rc = make_attn_tensor_map(&m.m32, base, DH, H, rows, frames, stride_r, stride_b, 16, box_rows, false);
  else m.m32 = m.m128;
  return rc;
}

// ---- host: what every attention entry point shares ----
// The head dims the attention kernels are instantiated for (include/motionclone_b200.h and ops.ATTN_HEAD_DIMS
// list the same set): calls f(std::integral_constant<int, DH>) and returns its status, MC_E_UNSUPPORTED for any other DH.
template <typename F>
inline int dispatch_head_dim(const char* entry, int DH, F&& f) {
  switch (DH) {
    case 8: return f(std::integral_constant<int, 8>{});
    case 16: return f(std::integral_constant<int, 16>{});
    case 32: return f(std::integral_constant<int, 32>{});
    case 40: return f(std::integral_constant<int, 40>{});
    case 64: return f(std::integral_constant<int, 64>{});
    case 80: return f(std::integral_constant<int, 80>{});
    case 160: return f(std::integral_constant<int, 160>{});
    default: break;
  }
  set_error("%s: unsupported head dim %d (8, 16, 32, 40, 64, 80, 160)", entry, DH);
  return MC_E_UNSUPPORTED;
}

// Argument checks, in the order the entry points apply them (checks of one kernel family go between the two calls):
// every pointer set and every dim positive (MC_E_INVALID) ...
inline int check_attn_operands(const char* entry, std::initializer_list<const void*> ptrs, std::initializer_list<int> dims) {
  bool ok = true;
  for (const void* p : ptrs) ok = ok && p != nullptr;
  for (int d : dims) ok = ok && d > 0;
  if (!ok) {
    set_error("%s: null pointer or non-positive dims", entry);
    return MC_E_INVALID;
  }
  return MC_OK;
}
// ... then B and H within the grid's y / z limit (MC_E_UNSUPPORTED), strides in multiples of 8 elements and 16-byte
// aligned pointers (MC_E_INVALID)
inline int check_attn_layout(const char* entry, int B, int H, std::initializer_list<int64_t> strides,
                             std::initializer_list<const void*> ptrs) {
  if (B > 65535 || H > 65535) {
    set_error("%s: B and H must be at most 65535", entry);
    return MC_E_UNSUPPORTED;
  }
  int64_t s_or = 0;
  uintptr_t p_or = 0;
  for (int64_t s : strides) s_or |= s;
  for (const void* p : ptrs) p_or |= (uintptr_t)p;
  if (s_or % 8 || p_or % 16) {
    set_error("%s: pointers must be 16-byte aligned and strides multiples of 8 elements", entry);
    return MC_E_INVALID;
  }
  return MC_OK;
}

// Grid (H, runs, B) of the cross-attention pair: a CTA takes a run of tiles_per_cta consecutive query tiles; enough CTAs
// for ~2 waves of (148 SMs x resident CTAs); K / V are re-read once per CTA, so longer runs amortise them
inline int xattn_grid(const char* entry, int n_tiles, int H, int B, int resident_ctas, int& tiles_per_cta, dim3& grid) {
  const int64_t tasks = (int64_t)n_tiles * H * B;
  int tpc = (int)(tasks / (148 * resident_ctas * 2));
  tpc = tpc < 1 ? 1 : (tpc > 8 ? 8 : tpc);
  const int runs = (n_tiles + tpc - 1) / tpc;
  if (runs > 65535) {
    set_error("%s: too many query tiles (%d)", entry, n_tiles);
    return MC_E_UNSUPPORTED;
  }
  tiles_per_cta = tpc;
  grid = dim3(H, runs, B);
  return MC_OK;
}

// ---- device: tensor-map load into shared memory, completion on an mbarrier ----
__device__ __forceinline__ void tma_load_4d(void* sdst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(sdst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

// one thread: issue the loads of one [ROWS][DH] tile (rows r0.. of head h, frame b); bytes = TileParts<DH, ROWS>::BYTES.
// The maps' box height must be ROWS.
template <int DH, int ROWS = 128>
__device__ __forceinline__ void tma_load_tile(uint8_t* sdst, const CUtensorMap* map128, const CUtensorMap* map32,
                                              uint64_t* bar, int r0, int h, int b) {
  using T = TileParts<DH, ROWS>;
#pragma unroll
  for (int p = 0; p < T::N64; ++p) tma_load_4d(sdst + T::part64_off(p), map128, bar, p * 64, h, r0, b);
#pragma unroll
  for (int p = 0; p < T::N16; ++p) tma_load_4d(sdst + T::part16_off(p), map32, bar, T::N64 * 64 + p * 16, h, r0, b);
}

// ---- swizzled shared-memory descriptors (cute::UMMA::SmemDescriptor, version 1) ----
//   layout_type [61,64): 2 = SWIZZLE_128B, 6 = SWIZZLE_32B
__device__ __forceinline__ uint64_t umma_desc_sw(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)layout << 61;
  return d;
}
// K-major SW128 part, k16 step ks (0..3): rows 128 B apart, 8-row groups 1024 B apart, 32 B per k step
__device__ __forceinline__ uint64_t desc_k128(uint32_t part_addr, int ks) {
  return umma_desc_sw(part_addr + ks * 32, 16, 1024, 2);
}
// K-major SW32 part (one k16 step): rows 32 B apart, 8-row groups 256 B apart
__device__ __forceinline__ uint64_t desc_k32(uint32_t part_addr) { return umma_desc_sw(part_addr, 16, 256, 6); }
// MN-major SW128 part, k16 step ks over the ROWS (16 rows = 2048 B): 8-row groups 1024 B apart; 64-element MN atoms
// `lbo_bytes` apart (only read when the MMA's M / N extent exceeds 64)
__device__ __forceinline__ uint64_t desc_mn128(uint32_t part_addr, int ks, uint32_t lbo_bytes = 16384) {
  return umma_desc_sw(part_addr + ks * 2048, lbo_bytes, 1024, 2);
}
// MN-major SW32 part (16 elements wide), k16 step ks over the rows (16 rows = 512 B): 8-row groups 256 B apart
__device__ __forceinline__ uint64_t desc_mn32(uint32_t part_addr, int ks) {
  return umma_desc_sw(part_addr + ks * 512, 4096, 256, 6);
}

// instruction descriptor with both majors selectable (bit 15: A is MN-major, bit 16: B is MN-major)
__device__ __forceinline__ uint32_t umma_idesc_f16(int M, int N, bool a_mn, bool b_mn) {
  uint32_t d = 0;
  d |= 1u << 4;  // fp32 accumulate
  d |= (a_mn ? 1u : 0u) << 15;
  d |= (b_mn ? 1u : 0u) << 16;
  d |= (uint32_t)(N >> 3) << 17;
  d |= (uint32_t)(M >> 4) << 24;
  return d;
}

// ---- single-thread MMA issue + commit, TMEM loads, tcgen05 fences ----
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accum)
      : "memory");
}

__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[AROWS x BROWS] (=)+= A[AROWS x DH] B[BROWS x DH]^T with both operands K-major tiles in shared memory (S = Q K^T,
// dP = dO V^T and their transposes): one MMA per k16 step over the head dim, SW128 parts first, then SW32 parts
template <int DH, int AROWS, int BROWS>
__device__ __forceinline__ void issue_kmajor(uint32_t d_tmem, uint32_t sA, uint32_t sB) {
  using TA = TileParts<DH, AROWS>;
  using TB = TileParts<DH, BROWS>;
  const uint32_t idesc = umma_idesc_f16(AROWS, BROWS, false, false);
  uint32_t acc = 0;
#pragma unroll
  for (int p = 0; p < TA::N64; ++p)
#pragma unroll
    for (int ks = 0; ks < TA::KS64; ++ks) {
      umma_f16(d_tmem, desc_k128(sA + TA::part64_off(p), ks), desc_k128(sB + TB::part64_off(p), ks), idesc, acc);
      acc = 1;
    }
#pragma unroll
  for (int p = 0; p < TA::N16; ++p) {
    umma_f16(d_tmem, desc_k32(sA + TA::part16_off(p)), desc_k32(sB + TB::part16_off(p)), idesc, acc);
    acc = 1;
  }
}

// byte offset of (row r, 16-byte chunk c of 8) inside a K-major SW128 part written by threads (P, dS tiles)
__device__ __forceinline__ uint32_t sw128_chunk_off(int r, int c) { return (uint32_t)(r * 128 + ((c ^ (r & 7)) << 4)); }

// ---- TMEM 32-column load / 16-column store (32x32b: thread = lane = row) ----
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
      "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(r[0]), "r"(r[1]),
               "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
// one row (DHP fp16, DHP % 16 == 0) of a K-major SW128 tile part in shared memory -> DHP / 2 packed TMEM columns of the
// calling thread's lane: how a resident [128][DH <= 48] operand tile becomes a tensor-memory A operand
template <int DHP>
__device__ __forceinline__ void smem_row_to_tmem(const uint8_t* part, int r, uint32_t taddr) {
  static_assert(DHP % 16 == 0 && DHP <= 64, "one SW128 part");
  uint32_t v[DHP / 2];
#pragma unroll
  for (int c = 0; c < DHP / 8; ++c) {
    const uint4 x = *reinterpret_cast<const uint4*>(part + sw128_chunk_off(r, c));
    v[4 * c] = x.x, v[4 * c + 1] = x.y, v[4 * c + 2] = x.z, v[4 * c + 3] = x.w;
  }
#pragma unroll
  for (int c = 0; c < DHP / 16; ++c) tmem_st8(taddr + c * 8, v + c * 8);
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
      "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
      "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]),
      "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
// D (+)= A B with A in TENSOR MEMORY (fp16 pairs: lane = row m, 32-bit column j = elements k = 2j, 2j + 1; 8 columns per
// k16 step) and B through a shared-memory descriptor: P / dS tiles never round-trip through shared memory.
__device__ __forceinline__ void umma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// D[128 x DH] (+)= A[128 x KROWS] B[KROWS x DH] (P V, dS K, P^T dO, dS^T Q): A = fp16 pairs in TENSOR MEMORY, k16 step ks
// at a_tmem(ks) (8 packed columns per step when contiguous); B = a KROWS-row tile read MN-major (its rows are the K
// dimension), so it needs no transpose. One MMA per (k16 step, part of B).
template <int DH, int KROWS, typename AddrFn>
__device__ __forceinline__ void issue_ts_mn(uint32_t d_tmem, AddrFn a_tmem, uint32_t sB, bool accumulate) {
  using T = TileParts<DH, KROWS>;
  const uint32_t idesc64 = umma_idesc_f16(128, T::W64, false, true);
  const uint32_t idesc16 = umma_idesc_f16(128, 16, false, true);
#pragma unroll
  for (int ks = 0; ks < KROWS / 16; ++ks) {
    const uint32_t a = a_tmem(ks);
    const uint32_t acc = (accumulate || ks > 0) ? 1u : 0u;
#pragma unroll
    for (int p = 0; p < T::N64; ++p) umma_f16_ts(d_tmem + p * 64, a, desc_mn128(sB + T::part64_off(p), ks), idesc64, acc);
#pragma unroll
    for (int p = 0; p < T::N16; ++p)
      umma_f16_ts(d_tmem + T::N64 * 64 + p * 16, a, desc_mn32(sB + T::part16_off(p), ks), idesc16, acc);
  }
}

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// exp2 of a PAIR on the FMA pipe (FADD2 / FFMA2, two fp32 lanes per instruction) instead of the 16-lane/clk MUFU: the
// attention kernels are bound by MUFU.EX2 issue, the FMA pipe idles, so a fixed fraction of the pairs goes this way.
// x = n + f with n = round(x) by the 1.5 * 2^23 trick (the integer lands in the low mantissa bits), 2^f on [-0.5, 0.5] by
// the degree-4 minimax polynomial (max relative error 2.7e-6, the probabilities are rounded to fp16, half-ulp 4.9e-4,
// right after; degree 3, 7.5e-5, moved the 32-frame extraction's top-1 agreement with the oracle measurably), 2^n by adding n << 23 to the exponent field. Inputs are clamped at -126 (result 2^-126: 0 in fp16).
__device__ __forceinline__ void ex2_poly_pair(float s0, float s1, float c, float negm, float& p0, float& p1) {
  uint64_t sp, cc, mm, x, t, f, p;
  asm("mov.b64 %0, {%1, %2};" : "=l"(sp) : "f"(s0), "f"(s1));
  asm("mov.b64 %0, {%1, %1};" : "=l"(cc) : "f"(c));
  asm("mov.b64 %0, {%1, %1};" : "=l"(mm) : "f"(negm));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(x) : "l"(sp), "l"(cc), "l"(mm));
  float x0, x1;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(x0), "=f"(x1) : "l"(x));
  x0 = fmaxf(x0, -126.f), x1 = fmaxf(x1, -126.f);
  asm("mov.b64 %0, {%1, %2};" : "=l"(x) : "f"(x0), "f"(x1));
  uint64_t magic, nmagic, k4, k3, k2, k1, k0;
  asm("mov.b64 %0, {%1, %1};" : "=l"(magic) : "f"(12582912.f));
  asm("mov.b64 %0, {%1, %1};" : "=l"(nmagic) : "f"(-12582912.f));
  asm("mov.b64 %0, {%1, %1};" : "=l"(k4) : "f"(0.009570101276040077f));
  asm("mov.b64 %0, {%1, %1};" : "=l"(k3) : "f"(0.05591786280274391f));
  asm("mov.b64 %0, {%1, %1};" : "=l"(k2) : "f"(0.240247443318367f));
  asm("mov.b64 %0, {%1, %1};" : "=l"(k1) : "f"(0.6931217908859253f));
  asm("mov.b64 %0, {%1, %1};" : "=l"(k0) : "f"(0.9999992847442627f));
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(t) : "l"(x), "l"(magic));
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(f) : "l"(t), "l"(nmagic));   // n = round(x)
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(f) : "l"(x), "l"(f));        // f = x - n
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(p) : "l"(k4), "l"(f), "l"(k3));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(p) : "l"(p), "l"(f), "l"(k2));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(p) : "l"(p), "l"(f), "l"(k1));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(p) : "l"(p), "l"(f), "l"(k0));
  float q0, q1, t0, t1;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(q0), "=f"(q1) : "l"(p));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(t0), "=f"(t1) : "l"(t));
  p0 = __uint_as_float(__float_as_uint(q0) + (__float_as_uint(t0) << 23));
  p1 = __uint_as_float(__float_as_uint(q1) + (__float_as_uint(t1) << 23));
}
// Every MC_EX2_POLY_PERIOD-th pair of an unrolled softmax loop takes the polynomial (0: none).
#ifndef MC_EX2_POLY_PERIOD
#define MC_EX2_POLY_PERIOD 4
#endif
__device__ __forceinline__ void ex2_pair(int pair_index, float s0, float s1, float c, float negm, float& p0, float& p1) {
  if (MC_EX2_POLY_PERIOD > 0 && pair_index % (MC_EX2_POLY_PERIOD > 0 ? MC_EX2_POLY_PERIOD : 1) == (MC_EX2_POLY_PERIOD - 1)) {
    ex2_poly_pair(s0, s1, c, negm, p0, p1);
  } else {
    p0 = ex2_approx(fmaf(s0, c, negm));
    p1 = ex2_approx(fmaf(s1, c, negm));
  }
}

template <int COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* slot) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "n"(COLS)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t base) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "n"(COLS) : "memory");
}

}  // namespace mc
