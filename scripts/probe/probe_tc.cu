// Hardware probes for the building blocks of csrc/spatial_attn_tc.cu (TEST / BRING-UP TOOL, not product code):
// each probe isolates one feature (tensor-map TMA with 128B / 32B swizzle, swizzled K-major / MN-major UMMA descriptors,
// MN-major A operands, tcgen05.st) and checks it against a CPU computation. One probe per process (a faulting probe must
// not poison the next):   probe_tc <name>      names: tma128 tma32 qk40 qk80 qk160 pv40 pv80 pv160 ts40 ts80 ts160 amn40 amn80 tmemst
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O2 -std=c++17 -I motionclone_b200/csrc scripts/probe/probe_tc.cu
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "tma_common.cuh"

namespace mc {  // host symbols mc_common.cuh declares
void set_error(const char*, ...) {}
void count_launch() {}
int check_launch(const char*) { return 0; }
}  // namespace mc
using namespace mc;

#define CK(x)                                                                      \
  do {                                                                             \
    cudaError_t e_ = (x);                                                          \
    if (e_ != cudaSuccess) {                                                       \
      printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); \
      exit(2);                                                                     \
    }                                                                              \
  } while (0)

static float h2f(__half h) { return __half2float(h); }

// ---- probe kernels -------------------------------------------------------------------------------------------------
__global__ void k_tma_dump(const __grid_constant__ CUtensorMap map, uint8_t* out, int bytes, int c0, int c1, int c2, int c3) {
  extern __shared__ uint8_t raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + 32768);
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    fence_mbar_init();
  }
  for (int i = threadIdx.x; i < bytes / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(smem)[i] = 0xdeadbeefu;
  fence_proxy_async();
  __syncthreads();
  if (threadIdx.x == 0) {
    mbar_arrive_expect_tx(bar, bytes);
    tma_load_4d(smem, &map, bar, c0, c1, c2, c3);
  }
  mbar_wait(bar, 0);
  for (int i = threadIdx.x; i < bytes; i += blockDim.x) out[i] = smem[i];
}

// mode 0: D[128x128] = A B^T, A/B = [128][DH] tiles by TMA (K-major)            -> out fp32 [128][128]
// mode 1: D[128xDHP] = P V, P [128][128] fp16 from global written by threads (K-major SW128), V tile by TMA (MN-major)
// mode 2: D[128xDHP] = A^T-as-MN-major . K : X^T [128 k][128 m] fp16 from global written by threads as a K-major SW128
//         tile of X^T (what the dK GEMM reads), read here as an MN-major A (what the dQ GEMM reads); B = K tile MN-major
template <int DH>
__global__ void __launch_bounds__(128) k_mma(const __grid_constant__ CUtensorMap ma128, const __grid_constant__ CUtensorMap ma32,
                                              const __grid_constant__ CUtensorMap mb128, const __grid_constant__ CUtensorMap mb32,
                                              const __half* pmat, float* out, int mode) {
  using T = TileParts<DH>;
  extern __shared__ uint8_t raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sA = smem;
  uint8_t* sB = smem + T::BYTES;
  uint8_t* sP = smem + 2 * T::BYTES;
  uint64_t* bar = reinterpret_cast<uint64_t*>(sP + 32768);
  uint64_t* bar2 = bar + 1;
  uint32_t* slot = reinterpret_cast<uint32_t*>(bar + 2);
  const int tid = threadIdx.x, warp = tid >> 5;
  if (warp == 0) tmem_alloc<512>(slot);
  if (tid == 0) {
    mbar_init(bar, 1), mbar_init(bar2, 1);
    fence_mbar_init();
  }
  if (mode >= 1 && mode != 3) {  // thread = row: write its 128 fp16 as two K-major SW128 parts
    const uint4* src = reinterpret_cast<const uint4*>(pmat + (size_t)tid * 128);
    for (int ch = 0; ch < 16; ++ch) *reinterpret_cast<uint4*>(sP + (ch >> 3) * 16384 + sw128_chunk_off(tid, ch & 7)) = src[ch];
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tb = *slot;
  if (mode == 3) {  // thread = row = TMEM lane: its 128 fp16 as 64 packed columns at [256, 320)
    const uint32_t* src = reinterpret_cast<const uint32_t*>(pmat + (size_t)tid * 128);
    uint32_t r[32];
    for (int half = 0; half < 2; ++half) {
      for (int i = 0; i < 32; ++i) r[i] = src[half * 32 + i];
      tmem_st32(tb + ((uint32_t)(warp * 32) << 16) + 256 + half * 32, r);
    }
    tmem_st_wait();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
  }
  if (tid == 0) {
    if (mode == 0) {
      mbar_arrive_expect_tx(bar, 2 * T::BYTES);
      tma_load_tile<DH>(sA, &ma128, &ma32, bar, 0, 1, 0);
      tma_load_tile<DH>(sB, &mb128, &mb32, bar, 0, 1, 0);
    } else {
      mbar_arrive_expect_tx(bar, T::BYTES);
      tma_load_tile<DH>(sB, &mb128, &mb32, bar, 0, 1, 0);
    }
    mbar_wait(bar, 0);
    tc_fence_after();
    if (mode == 0) {
      // S tile exactly as the forward kernel issues it
      const uint32_t idesc = umma_idesc_f16(128, 128, false, false);
      uint32_t acc = 0;
      for (int p = 0; p < T::N64; ++p)
        for (int ks = 0; ks < T::KS64; ++ks) {
          umma_f16(tb, desc_k128(smem_u32(sA) + T::part64_off(p), ks), desc_k128(smem_u32(sB) + T::part64_off(p), ks), idesc, acc);
          acc = 1;
        }
      for (int p = 0; p < T::N16; ++p) {
        umma_f16(tb, desc_k32(smem_u32(sA) + T::part16_off(p)), desc_k32(smem_u32(sB) + T::part16_off(p)), idesc, acc);
        acc = 1;
      }
    } else if (mode == 3) {
      const uint32_t id64 = umma_idesc_f16(128, T::W64, false, true);
      const uint32_t id16 = umma_idesc_f16(128, 16, false, true);
      for (int ks = 0; ks < 8; ++ks) {
        const uint32_t a = tb + 256 + ks * 8;  // 8 packed columns per k16 step
        const uint32_t acc = ks > 0;
        for (int p = 0; p < T::N64; ++p) umma_f16_ts(tb + p * 64, a, desc_mn128(smem_u32(sB) + T::part64_off(p), ks), id64, acc);
        for (int p = 0; p < T::N16; ++p) umma_f16_ts(tb + T::N64 * 64 + p * 16, a, desc_mn32(smem_u32(sB) + T::part16_off(p), ks), id16, acc);
      }
    } else {
      const uint32_t id64 = umma_idesc_f16(128, T::W64, mode == 2, true);
      const uint32_t id16 = umma_idesc_f16(128, 16, mode == 2, true);
      for (int ks = 0; ks < 8; ++ks) {
        // mode 1: A K-major, k16 step ks = keys [16 ks, 16 ks + 16): part ks>>2, 32 B per step
        // mode 2: A MN-major over the SAME bytes: rows of the stored tile are the K dimension (16 rows = 2048 B per step),
        //         the two 64-wide parts are the M atoms (LBO = 16384)
        const uint64_t a = mode == 1 ? desc_k128(smem_u32(sP) + (ks >> 2) * 16384, ks & 3) : desc_mn128(smem_u32(sP), ks, 16384);
        const uint32_t acc = ks > 0;
        for (int p = 0; p < T::N64; ++p) umma_f16(tb + p * 64, a, desc_mn128(smem_u32(sB) + T::part64_off(p), ks), id64, acc);
        for (int p = 0; p < T::N16; ++p) umma_f16(tb + T::N64 * 64 + p * 16, a, desc_mn32(smem_u32(sB) + T::part16_off(p), ks), id16, acc);
      }
    }
    umma_commit(bar2);
  }
  mbar_wait(bar2, 0);
  tc_fence_after();
  const uint32_t la = tb + ((uint32_t)(warp * 32) << 16);
  const int ncol = mode == 0 ? 128 : T::DHP;
  for (int c = 0; c < ncol; c += 16) {
    uint32_t r[16];
    tmem_ld16(la + c, r);
    tmem_ld_wait();
    for (int i = 0; i < 16; ++i) out[(size_t)tid * ncol + c + i] = __uint_as_float(r[i]);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc<512>(tb);
}

__global__ void __launch_bounds__(128) k_tmemst(float* out) {
  __shared__ uint32_t slot;
  const int tid = threadIdx.x, warp = tid >> 5;
  if (warp == 0) tmem_alloc<64>(&slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t la = slot + ((uint32_t)(warp * 32) << 16);
  uint32_t r[16];
  for (int i = 0; i < 16; ++i) r[i] = __float_as_uint((float)(tid * 100 + i));
  tmem_st16(la + 16, r);
  tmem_st_wait();
  uint32_t q[16];
  tmem_ld16(la + 16, q);
  tmem_ld_wait();
  for (int i = 0; i < 16; ++i) q[i] = __float_as_uint(__uint_as_float(q[i]) * 0.5f);
  tmem_st16(la + 16, q);
  tmem_st_wait();
  tmem_ld16(la + 16, r);
  tmem_ld_wait();
  for (int i = 0; i < 16; ++i) out[tid * 16 + i] = __uint_as_float(r[i]);
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc<64>(slot);
}

// ---- host ----------------------------------------------------------------------------------------------------------
struct Synth {
  int N, H, DH, B;
  int64_t sr, sb;
  std::vector<__half> data;  // fused [B][N][3][H][DH]
  __half* dev = nullptr;
  Synth(int N_, int H_, int DH_, int B_) : N(N_), H(H_), DH(DH_), B(B_) {
    sr = 3 * H * DH, sb = (int64_t)N * sr;
    data.resize((size_t)B * sb);
    uint32_t s = 12345u + DH;
    for (auto& x : data) {
      s = s * 1664525u + 1013904223u;
      x = __float2half(((int)((s >> 9) & 0xff) - 128) / 64.0f);
    }
    CK(cudaMalloc(&dev, data.size() * 2));
    CK(cudaMemcpy(dev, data.data(), data.size() * 2, cudaMemcpyHostToDevice));
  }
  float at(int which, int b, int r, int h, int e) const {
    if (r >= N || e >= DH) return 0.f;
    return h2f(data[(size_t)b * sb + (size_t)r * sr + (size_t)which * H * DH + h * DH + e]);
  }
  const __half* ptr(int which) const { return dev + (size_t)which * H * DH; }
};

static int run_tma(bool sw128) {
  const int DH = sw128 ? 40 : 80;
  Synth t(200, 2, DH, 2);
  CUtensorMap map;
  if (make_attn_tensor_map(&map, t.ptr(1), DH, 2, 200, 2, t.sr, t.sb, sw128 ? 64 : 16, 128, sw128)) {
    printf("encode failed\n");
    return 1;
  }
  const int bytes = sw128 ? 16384 : 4096;
  uint8_t* dout;
  CK(cudaMalloc(&dout, bytes));
  CK(cudaFuncSetAttribute(k_tma_dump, cudaFuncAttributeMaxDynamicSharedMemorySize, 40000));
  const int e0 = sw128 ? 0 : 64;
  k_tma_dump<<<1, 128, 40000>>>(map, dout, bytes, e0, 1, 128, 1);
  CK(cudaDeviceSynchronize());
  std::vector<uint8_t> hb(bytes);
  CK(cudaMemcpy(hb.data(), dout, bytes, cudaMemcpyDeviceToHost));
  const __half* hh = reinterpret_cast<const __half*>(hb.data());
  int bad = 0;
  const int rowb = sw128 ? 128 : 32, nch = sw128 ? 8 : 2;
  for (int r = 0; r < 128; ++r)
    for (int c = 0; c < nch; ++c) {
      const int off = sw128 ? r * 128 + ((c ^ (r & 7)) << 4) : r * 32 + ((c ^ ((r >> 2) & 1)) << 4);
      for (int i = 0; i < 8; ++i) {
        const float want = t.at(1, 1, 128 + r, 1, e0 + c * 8 + i);
        const float got = h2f(hh[off / 2 + i]);
        if (want != got && bad++ < 5) printf("  mismatch r=%d c=%d i=%d want %f got %f\n", r, c, i, want, got);
      }
    }
  (void)rowb;
  printf("PROBE %s: %s (%d bad)\n", sw128 ? "tma128" : "tma32", bad ? "FAIL" : "PASS", bad);
  return bad != 0;
}

template <int DH>
static int run_mma(int mode, const char* name) {
  using T = TileParts<DH>;
  Synth t(128, 2, DH, 1);
  CUtensorMap a128, a32, b128, b32;
  const int wa = 0, wb = mode == 0 ? 1 : (mode == 2 ? 1 : 2);  // mode0: Q,K  mode1/3: V  mode2: K
  int rc = make_attn_tensor_map(&a128, t.ptr(wa), DH, 2, 128, 1, t.sr, t.sb, 64, 128, true);
  rc |= make_attn_tensor_map(&b128, t.ptr(wb), DH, 2, 128, 1, t.sr, t.sb, 64, 128, true);
  a32 = a128, b32 = b128;
  if (T::N16 > 0) {
    rc |= make_attn_tensor_map(&a32, t.ptr(wa), DH, 2, 128, 1, t.sr, t.sb, 16, 128, false);
    rc |= make_attn_tensor_map(&b32, t.ptr(wb), DH, 2, 128, 1, t.sr, t.sb, 16, 128, false);
  }
  if (rc) {
    printf("encode failed\n");
    return 1;
  }
  std::vector<__half> P(128 * 128);
  uint32_t s = 777;
  for (auto& x : P) {
    s = s * 1664525u + 1013904223u;
    x = __float2half(((int)((s >> 10) & 0x3f) - 32) / 32.0f);
  }
  __half* dP;
  CK(cudaMalloc(&dP, P.size() * 2));
  CK(cudaMemcpy(dP, P.data(), P.size() * 2, cudaMemcpyHostToDevice));
  const int ncol = mode == 0 ? 128 : T::DHP;
  float* dout;
  CK(cudaMalloc(&dout, 128 * ncol * 4));
  const int smem = 2 * T::BYTES + 32768 + 64 + 1024;
  CK(cudaFuncSetAttribute(k_mma<DH>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  k_mma<DH><<<1, 128, smem>>>(a128, a32, b128, b32, dP, dout, mode);
  CK(cudaDeviceSynchronize());
  std::vector<float> out(128 * ncol);
  CK(cudaMemcpy(out.data(), dout, out.size() * 4, cudaMemcpyDeviceToHost));
  double maxerr = 0;
  for (int m = 0; m < 128; ++m)
    for (int n = 0; n < ncol; ++n) {
      double want = 0;
      if (mode == 0) {
        for (int e = 0; e < DH; ++e) want += (double)t.at(0, 0, m, 1, e) * t.at(1, 0, n, 1, e);
      } else if (mode == 1 || mode == 3) {
        for (int j = 0; j < 128; ++j) want += (double)h2f(P[m * 128 + j]) * t.at(2, 0, j, 1, n);
      } else {  // D[m][n] = sum_k X^T[k][m] * K[k][n]
        for (int j = 0; j < 128; ++j) want += (double)h2f(P[j * 128 + m]) * t.at(1, 0, j, 1, n);
      }
      const double err = fabs(want - out[m * ncol + n]);
      if (err > maxerr) maxerr = err;
    }
  const bool ok = maxerr < 2e-2;
  printf("PROBE %s: %s (max abs err %.3e)\n", name, ok ? "PASS" : "FAIL", maxerr);
  if (!ok) {
    printf("  first row got : ");
    for (int n = 0; n < 8; ++n) printf("%8.3f ", out[n]);
    printf("\n");
  }
  return !ok;
}

static int run_tmemst() {
  float* d;
  CK(cudaMalloc(&d, 128 * 16 * 4));
  k_tmemst<<<1, 128>>>(d);
  CK(cudaDeviceSynchronize());
  std::vector<float> o(128 * 16);
  CK(cudaMemcpy(o.data(), d, o.size() * 4, cudaMemcpyDeviceToHost));
  int bad = 0;
  for (int t = 0; t < 128; ++t)
    for (int i = 0; i < 16; ++i) bad += o[t * 16 + i] != 0.5f * (t * 100 + i);
  printf("PROBE tmemst: %s (%d bad)\n", bad ? "FAIL" : "PASS", bad);
  return bad != 0;
}

int main(int argc, char** argv) {
  const std::string n = argc > 1 ? argv[1] : "";
  if (n == "tma128") return run_tma(true);
  if (n == "tma32") return run_tma(false);
  if (n == "qk40") return run_mma<40>(0, "qk40");
  if (n == "qk80") return run_mma<80>(0, "qk80");
  if (n == "qk160") return run_mma<160>(0, "qk160");
  if (n == "qk16") return run_mma<16>(0, "qk16");
  if (n == "pv40") return run_mma<40>(1, "pv40");
  if (n == "pv80") return run_mma<80>(1, "pv80");
  if (n == "pv160") return run_mma<160>(1, "pv160");
  if (n == "pv16") return run_mma<16>(1, "pv16");
  if (n == "ts40") return run_mma<40>(3, "ts40");
  if (n == "ts80") return run_mma<80>(3, "ts80");
  if (n == "ts160") return run_mma<160>(3, "ts160");
  if (n == "amn40") return run_mma<40>(2, "amn40");
  if (n == "amn80") return run_mma<80>(2, "amn80");
  if (n == "tmemst") return run_tmemst();
  printf("unknown probe '%s'\n", n.c_str());
  return 3;
}
