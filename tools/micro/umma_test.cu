// Micro-validation of the tcgen05 primitives the tensor-core NDE kernel is built from (sm_100a only).
//   T1  SS  kind::tf32, M=128, N=32, K=96: A K-major (LBO=128, SBO=3072), B K-major padded (SBO=128, LBO=528)
//   T2  TS  same product with A staged in TMEM by tcgen05.st (lane = row, column = k)
//   T3  SS  quadrant placement: A descriptor start moved back by q*4*SBO so a 32-row A lands in TMEM lanes 32q..32q+31
//   T4  3xTF32 accuracy on random FP32 data (hi/lo split, three accumulating MMAs)
//   T5  timings (clock64): MMA chains at N=16/32 (SS and TS), TS at N=16/32/48/64, commit->mbarrier round trip, tcgen05.ld
//   T8  address probe of the N=48 B plane of the forward kernel's layers 2/3 (SBO=128, LBO=6*128+16=784), checked on the host
// build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o umma_test umma_test.cu
#include <cuda_runtime.h>
#include <stdint.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e), __FILE__, __LINE__); exit(1);} } while (0)

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo >> 4) & 0x3FFF) << 16) | ((uint64_t)((sbo >> 4) & 0x3FFF) << 32) |
         (1ull << 46);
}
__host__ __device__ constexpr uint32_t make_idesc(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void mma_ss(uint32_t d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d),
               "l"(a), "l"(b), "r"(idesc), "r"(acc)
               : "memory");
}
__device__ __forceinline__ void mma_ts(uint32_t d, uint32_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d),
               "r"(a), "l"(b), "r"(idesc), "r"(acc)
               : "memory");
}
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "W_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra W_DONE;\n\t"
      "bra W_LOOP;\n\t"
      "W_DONE:\n\t}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void fence_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const float* v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(__float_as_uint(v[0])),
               "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])),
               "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7]))
               : "memory");
}

// canonical no-swizzle K-major offsets (bytes) for 4-byte elements
__host__ __device__ inline uint32_t kmaj_off(int r, int k, uint32_t sbo, uint32_t lbo) {
  return (uint32_t)(r / 8) * sbo + (uint32_t)(k / 4) * lbo + (uint32_t)(r % 8) * 16 + (uint32_t)(k % 4) * 4;
}

constexpr int M_ = 128, K_ = 96;
constexpr uint32_t A_LBO = 128, A_SBO = (K_ / 4) * 128;  // 3072
constexpr uint32_t A_BYTES = (M_ / 8) * A_SBO;           // 49152
constexpr uint32_t B_SBO = 128;
__host__ __device__ constexpr uint32_t b_lbo(int N) { return (uint32_t)(N / 8) * 128 + 16; }
__host__ __device__ constexpr uint32_t b_bytes(int N, int K) { return (uint32_t)(K / 4) * b_lbo(N); }

struct Out {
  float d1[128 * 32];   // T1
  float d2[128 * 32];   // T2
  float d3[128 * 32];   // T3: three nets, net q in lanes 32q.., columns 0..15 of region q -> stored [lane][q*... ] see below
  float d4[128 * 32];   // T4
  long long t[32];
};

// Ahi/Alo: [128][96] row-major (m,k). Bhi/Blo: [32][96] (n,k). A3: [3][32][24]; B3: [16][24]
__global__ void __launch_bounds__(128, 1) umma_kernel(const float* __restrict__ A, const float* __restrict__ B,
                                                     const float* __restrict__ Ar, const float* __restrict__ Br,
                                                     const float* __restrict__ A3, const float* __restrict__ B3, Out* out, int test, int variant) {
  extern __shared__ __align__(1024) uint8_t sm[];
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // smem map
  uint8_t* sA = sm;                            // 49152 (hi)
  uint8_t* sA2 = sm + A_BYTES;                 // 49152 (lo)
  uint8_t* sB = sm + 2 * A_BYTES;              // N=32,K=96: 24*528 = 12672 (hi)
  uint8_t* sB2 = sB + 12800;                   // lo
  uint8_t* sA3 = sB2 + 12800;                  // 3 nets x (4 row groups x 768) = 9216 ; placed after 2*A -> plenty of room before it
  uint8_t* sB3 = sA3 + 9216;                   // N=16,K=24: 6 chunks x 272 = 1632
  if (tid == 0) {
    mbar_init(&bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  // zero all dynamic smem
  for (int i = tid; i < (int)((2 * A_BYTES + 2 * 12800 + 9216 + 8192) / 4); i += 128) reinterpret_cast<float*>(sm)[i] = 0.f;
  tc_before();
  __syncthreads();
  tc_after();
  const uint32_t tb = tmem_base_s;
  uint32_t parity = 0;
  // ---------------- T1: SS exact ----------------
  if (test == 1) {
  for (int i = tid; i < M_ * K_; i += 128) {
    const int m = i / K_, k = i % K_;
    *reinterpret_cast<float*>(sA + kmaj_off(m, k, A_SBO, A_LBO)) = A[i];
  }
  for (int i = tid; i < 32 * K_; i += 128) {
    const int n = i / K_, k = i % K_;
    *reinterpret_cast<float*>(sB + kmaj_off(n, k, B_SBO, b_lbo(32))) = B[i];
  }
  fence_async();
  __syncthreads();
  const uint32_t D1 = tb + 384;
  if (tid == 0) {
    tc_after();
    const uint32_t id = make_idesc(128, 32);
    for (int s = 0; s < K_ / 8; ++s) {
      const uint64_t ad = make_desc(smem_u32(sA) + s * 2 * A_LBO, A_LBO, A_SBO);
      const uint64_t bd = make_desc(smem_u32(sB) + s * 2 * b_lbo(32), b_lbo(32), B_SBO);
      mma_ss(D1, ad, bd, id, s > 0);
    }
    mma_commit(&bar);
  }
  mbar_wait(&bar, parity); parity ^= 1;
  tc_after();
  {
    float v[32];
    tmem_ld32(D1 + ((uint32_t)(warp * 32) << 16), v);
    for (int n = 0; n < 32; ++n) out->d1[(warp * 32 + lane) * 32 + n] = v[n];
  }
  tc_before();
  __syncthreads();
  }
  // ---------------- T2: TS (A in TMEM columns 0..95) ----------------
  if (test == 2) {
  for (int i = tid; i < 32 * K_; i += 128) {
    const int n = i / K_, k = i % K_;
    *reinterpret_cast<float*>(sB + kmaj_off(n, k, B_SBO, b_lbo(32))) = B[i];
  }
  fence_async();
  {
    const int m = warp * 32 + lane;
    for (int k0 = 0; k0 < K_; k0 += 8) {
      float v[8];
      for (int j = 0; j < 8; ++j) v[j] = A[m * K_ + k0 + j];
      tmem_st8(tb + ((uint32_t)(warp * 32) << 16) + k0, v);
    }
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  }
  tc_before();
  __syncthreads();
  const uint32_t D2 = tb + 416;
  if (tid == 0) {
    tc_after();
    const uint32_t id = make_idesc(128, 32);
    for (int s = 0; s < K_ / 8; ++s) {
      const uint64_t bd = make_desc(smem_u32(sB) + s * 2 * b_lbo(32), b_lbo(32), B_SBO);
      mma_ts(D2, tb + 8 * s, bd, id, s > 0);
    }
    mma_commit(&bar);
  }
  mbar_wait(&bar, parity); parity ^= 1;
  tc_after();
  {
    float v[32];
    tmem_ld32(D2 + ((uint32_t)(warp * 32) << 16), v);
    for (int n = 0; n < 32; ++n) out->d2[(warp * 32 + lane) * 32 + n] = v[n];
  }
  tc_before();
  __syncthreads();
  }
  // ---------------- T3: stacked nets, N=16, K=24 ----------------
  if (test == 3) {
  constexpr uint32_t A3_SBO = 6 * 128, A3_LBO = 128;
  for (int i = tid; i < 3 * 32 * 24; i += 128) {
    const int q = i / (32 * 24), r = (i / 24) % 32, k = i % 24;
    *reinterpret_cast<float*>(sA3 + q * 4 * A3_SBO + kmaj_off(r, k, A3_SBO, A3_LBO)) = A3[i];
  }
  for (int i = tid; i < 16 * 24; i += 128) {
    const int n = i / 24, k = i % 24;
    *reinterpret_cast<float*>(sB3 + kmaj_off(n, k, B_SBO, b_lbo(16))) = B3[i];
  }
  fence_async();
  __syncthreads();
  const uint32_t D3 = tb + 448;
  if (tid == 0) {
    tc_after();
    const uint32_t id = make_idesc(128, 16);
    for (int q = 0; q < 3; ++q)
      for (int s = 0; s < 3; ++s) {
        // net q's 32 rows must appear as rows 32q..32q+31: start = (its base) - q*4*SBO
        const uint32_t a0 = smem_u32(sA3) + s * 2 * A3_LBO;  // nets stacked in M: row m = net m/32, row m%32
        const uint64_t ad = make_desc(a0, A3_LBO, A3_SBO);
        const uint64_t bd = make_desc(smem_u32(sB3) + s * 2 * b_lbo(16), b_lbo(16), B_SBO);
        mma_ss(D3 + 16 * q, ad, bd, id, s > 0);
      }
    mma_commit(&bar);
  }
  mbar_wait(&bar, parity); parity ^= 1;
  tc_after();
  {
    float v[32];
    tmem_ld32(D3 + ((uint32_t)(warp * 32) << 16), v);  // columns 0..47 hold 3 regions; read 32 here (regions 0,1)
    for (int n = 0; n < 32; ++n) out->d3[(warp * 32 + lane) * 32 + n] = v[n];
  }
  tc_before();
  __syncthreads();
  }
  // ---------------- T4: 3xTF32 random, N=32, K=96 ----------------
  long long t0 = 0, t1 = 0;
  const uint32_t D4 = tb + 384;
  if (test == 4) {
  for (int i = tid; i < M_ * K_; i += 128) {
    const int m = i / K_, k = i % K_;
    const float x = Ar[i];
    uint32_t hb_;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hb_) : "f"(x));
    const float hi = __uint_as_float(hb_);
    *reinterpret_cast<float*>(sA + kmaj_off(m, k, A_SBO, A_LBO)) = hi;
    *reinterpret_cast<float*>(sA2 + kmaj_off(m, k, A_SBO, A_LBO)) = x - hi;
  }
  for (int i = tid; i < 32 * K_; i += 128) {
    const int n = i / K_, k = i % K_;
    const float x = Br[i];
    uint32_t hb_;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hb_) : "f"(x));
    const float hi = __uint_as_float(hb_);
    *reinterpret_cast<float*>(sB + kmaj_off(n, k, B_SBO, b_lbo(32))) = hi;
    *reinterpret_cast<float*>(sB2 + kmaj_off(n, k, B_SBO, b_lbo(32))) = x - hi;
  }
  fence_async();
  __syncthreads();
  if (tid == 0) {
    tc_after();
    const uint32_t id = make_idesc(128, 32);
    t0 = clock64();
    int first = 1;
    for (int term = 0; term < 3; ++term) {
      const uint8_t* a = term == 0 ? sA2 : sA;   // lo*hi, hi*lo, hi*hi
      const uint8_t* b = term == 1 ? sB2 : sB;
      for (int s = 0; s < K_ / 8; ++s) {
        mma_ss(D4, make_desc(smem_u32(a) + s * 2 * A_LBO, A_LBO, A_SBO), make_desc(smem_u32(b) + s * 2 * b_lbo(32), b_lbo(32), B_SBO), id,
               !first);
        first = 0;
      }
    }
    mma_commit(&bar);
  }
  mbar_wait(&bar, parity); parity ^= 1;
  if (tid == 0) { t1 = clock64(); out->t[0] = t1 - t0; }  // 36 SS MMAs N=32
  tc_after();
  {
    float v[32];
    tmem_ld32(D4 + ((uint32_t)(warp * 32) << 16), v);
    for (int n = 0; n < 32; ++n) out->d4[(warp * 32 + lane) * 32 + n] = v[n];
  }
  tc_before();
  __syncthreads();
  }
  // ---------------- T6: TS with MN-major B ([column block of 4][row][4]), N=16, arbitrary K window start ----------------
  if (test == 6) {
    const int ROWS = 160, KST = 50, KW = 56;   // window rows 50..105 of a 160-row operand
    // A (TMEM cols 0..55): A[m][kk] = A[m*96 + kk] ; B rows: Bv[n][row] = B[(n%32)*96 + (row % 96)] for n < 16
    {
      const int m = warp * 32 + lane;
      for (int k0 = 0; k0 < KW; k0 += 8) {
        float v[8];
        for (int j = 0; j < 8; ++j) v[j] = A[m * K_ + k0 + j];
        tmem_st8(tb + ((uint32_t)(warp * 32) << 16) + k0, v);
      }
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    }
    for (int i = tid; i < 16 * ROWS; i += 128) {
      const int n = i / ROWS, row = i % ROWS;
      *reinterpret_cast<float*>(sB + (n / 4) * ROWS * 16 + row * 16 + (n % 4) * 4) = B[n * K_ + (row % K_)];
    }
    fence_async();
    tc_before();
    __syncthreads();
    const uint32_t D6 = tb + 400;
    if (warp == 0) {
      tc_after();
      uint32_t el = 0;
      asm volatile("{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\telect.sync rx|px, 0xffffffff;\n\t@px mov.s32 %0, 1;\n\t}" : "+r"(el));
      if (el) {
        const uint32_t id = make_idesc(128, 16) | (1u << 16);  // B MN-major
        const uint64_t bd = (uint64_t)(((smem_u32(sB) + KST * 16) >> 4) & 0x3FFF) | ((uint64_t)((variant == 0 ? 128u : (uint32_t)ROWS * 16u) >> 4) << 16) | ((uint64_t)((variant == 0 ? (uint32_t)ROWS * 16u : 128u) >> 4) << 32) | (1ull << 46);
        for (int s = 0; s < KW / 8; ++s) mma_ts(D6, tb + 8 * s, bd + 8 * s, id, s > 0);
        mma_commit(&bar);
      }
      __syncwarp();
    }
    mbar_wait(&bar, parity); parity ^= 1;
    tc_after();
    {
      float v[32];
      tmem_ld32(D6 + ((uint32_t)(warp * 32) << 16), v);
      for (int n = 0; n < 32; ++n) out->d1[(warp * 32 + lane) * 32 + n] = v[n];
    }
    tc_before();
    __syncthreads();
  }
  // ---------------- T7: address probe. A = 8x8 identity (other rows 0), smem word i holds float(i): D[m][n] = word index of B(n, k=m)
  if (test == 7) {
    {
      const int m = warp * 32 + lane;
      float v[8];
      for (int j = 0; j < 8; ++j) v[j] = (m == j) ? 1.f : 0.f;
      tmem_st8(tb + ((uint32_t)(warp * 32) << 16), v);
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    }
    for (int i = tid; i < 8192; i += 128) reinterpret_cast<float*>(sB)[i] = (float)i;
    fence_async();
    tc_before();
    __syncthreads();
    const uint32_t D7 = tb + 400;
    if (warp == 0) {
      tc_after();
      uint32_t el = 0;
      asm volatile("{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\telect.sync rx|px, 0xffffffff;\n\t@px mov.s32 %0, 1;\n\t}" : "+r"(el));
      if (el) {
        const uint32_t id = make_idesc(128, 16) | ((variant & 1) ? (1u << 16) : 0u);
        const uint32_t lbo = 2048, sbo = 512;
        const uint64_t bd = (uint64_t)((smem_u32(sB) >> 4) & 0x3FFF) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) | (1ull << 46);
        mma_ts(D7, tb, bd, id, 0);
        mma_commit(&bar);
      }
      __syncwarp();
    }
    mbar_wait(&bar, parity); parity ^= 1;
    tc_after();
    {
      float v[32];
      tmem_ld32(D7 + ((uint32_t)(warp * 32) << 16), v);
      for (int n = 0; n < 32; ++n) out->d1[(warp * 32 + lane) * 32 + n] = v[n];
    }
    tc_before();
    __syncthreads();
  }
  // ---------------- T8: the same probe at N=48 with the layer-2/3 B plane of the forward kernel (SBO=128, LBO=784)
  if (test == 8) {
    {
      const int m = warp * 32 + lane;
      float v[8];
      for (int j = 0; j < 8; ++j) v[j] = (m == j) ? 1.f : 0.f;
      tmem_st8(tb + ((uint32_t)(warp * 32) << 16), v);
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    }
    for (int i = tid; i < 8192; i += 128) reinterpret_cast<float*>(sB)[i] = (float)i;
    fence_async();
    tc_before();
    __syncthreads();
    const uint32_t D8 = tb + 400;
    if (warp == 0) {
      tc_after();
      uint32_t el = 0;
      asm volatile("{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\telect.sync rx|px, 0xffffffff;\n\t@px mov.s32 %0, 1;\n\t}" : "+r"(el));
      if (el) { mma_ts(D8, tb, make_desc(smem_u32(sB), b_lbo(48), B_SBO), make_idesc(128, 48), 0); mma_commit(&bar); }
      __syncwarp();
    }
    mbar_wait(&bar, parity); parity ^= 1;
    tc_after();
    {
      float v[32];
      tmem_ld32(D8 + ((uint32_t)(warp * 32) << 16), v);
      for (int n = 0; n < 32; ++n) out->d1[(warp * 32 + lane) * 32 + n] = v[n];
      tmem_ld32(D8 + 32 + ((uint32_t)(warp * 32) << 16), v);
      for (int n = 0; n < 32; ++n) out->d2[(warp * 32 + lane) * 32 + n] = v[n];
    }
    tc_before();
    __syncthreads();
  }
  // ---------------- T5: timings (warp-uniform issue + elect.sync, descriptors advanced by adds) ----------------
  if (test == 5) {
  if (warp == 0) {
    tc_after();
    uint32_t el = 0;
    asm volatile("{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\telect.sync rx|px, 0xffffffff;\n\t@px mov.s32 %0, 1;\n\t}" : "+r"(el));
    const uint64_t ad0 = make_desc(smem_u32(sA), A_LBO, A_SBO);
    const uint64_t bd0 = make_desc(smem_u32(sB), b_lbo(32), B_SBO);
    const uint64_t astep = (2 * A_LBO) >> 4, bstep = (2 * b_lbo(32)) >> 4;
#define TIME_CHAIN(slot, REPS, NN, TS)                                                      \
    {                                                                                       \
      const uint32_t id = make_idesc(128, NN);                                              \
      long long c0 = clock64();                                                             \
      if (el) {                                                                             \
        for (int r = 0; r < REPS; ++r) {                                                    \
          _Pragma("unroll") for (int s = 0; s < 12; ++s) {                                  \
            if (TS) mma_ts(D4, tb + 8 * s, bd0 + s * bstep, id, 1);                         \
            else mma_ss(D4, ad0 + s * astep, bd0 + s * bstep, id, 1);                       \
          }                                                                                 \
        }                                                                                   \
        mma_commit(&bar);                                                                   \
      }                                                                                     \
      __syncwarp();                                                                         \
      long long c1 = clock64();                                                             \
      mbar_wait(&bar, parity); parity ^= 1;                                                 \
      long long c2 = clock64();                                                             \
      if (lane == 0) { out->t[slot] = c2 - c0; out->t[slot + 16] = c1 - c0; }              \
    }
    TIME_CHAIN(1, 6, 32, 0)
    TIME_CHAIN(2, 6, 32, 1)
    TIME_CHAIN(3, 6, 16, 0)
    TIME_CHAIN(4, 6, 16, 1)
    TIME_CHAIN(5, 12, 16, 1)
    TIME_CHAIN(6, 12, 32, 1)
    TIME_CHAIN(7, 12, 64, 1)
    TIME_CHAIN(9, 12, 48, 1)
    {
      const uint32_t id = make_idesc(128, 16);
      long long c0 = clock64();
      if (el) { mma_ts(D4, tb, bd0, id, 1); mma_commit(&bar); }
      __syncwarp();
      mbar_wait(&bar, parity); parity ^= 1;
      if (lane == 0) out->t[0] = clock64() - c0;
    }
    tc_before();
  } else { parity ^= 0; }
  __syncthreads();
  tc_after();
  // (9) tcgen05.ld x32 + wait, per warp (warp 0 reports)
  {
    float v[32];
    long long a0 = clock64();
    tmem_ld32(D4 + ((uint32_t)(warp * 32) << 16), v);
    long long a1 = clock64();
    float s = 0.f;
    for (int i = 0; i < 32; ++i) s += v[i];
    if (tid == 0) out->t[8] = a1 - a0;
    if (s == 123.456f) out->d1[0] = 1;
  }
  }
  tc_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tb), "r"(512));
}

static float tf32_rna(float x) {
  uint32_t u;
  memcpy(&u, &x, 4);
  u += 0x1000u;
  u &= 0xFFFFE000u;
  float r;
  memcpy(&r, &u, 4);
  return r;
}

int main(int argc, char** argv) {
  const int test = argc > 1 ? atoi(argv[1]) : 1;
  std::vector<float> A(128 * 96), B(32 * 96), Ar(128 * 96), Br(32 * 96), A3(3 * 32 * 24), B3(16 * 24);
  srand(1);
  for (auto& x : A) x = (float)((rand() % 17) - 8) / 8.f;
  for (auto& x : B) x = (float)((rand() % 17) - 8) / 4.f;
  for (auto& x : Ar) x = (float)rand() / RAND_MAX - 0.5f;
  for (auto& x : Br) x = (float)rand() / RAND_MAX - 0.5f;
  for (auto& x : A3) x = (float)((rand() % 9) - 4) / 4.f;
  for (auto& x : B3) x = (float)((rand() % 9) - 4) / 2.f;
  float *dA, *dB, *dAr, *dBr, *dA3, *dB3;
  Out* dout;
  CK(cudaMalloc(&dA, A.size() * 4)); CK(cudaMalloc(&dB, B.size() * 4)); CK(cudaMalloc(&dAr, Ar.size() * 4));
  CK(cudaMalloc(&dBr, Br.size() * 4)); CK(cudaMalloc(&dA3, A3.size() * 4)); CK(cudaMalloc(&dB3, B3.size() * 4));
  CK(cudaMalloc(&dout, sizeof(Out)));
  CK(cudaMemset(dout, 0, sizeof(Out)));
  CK(cudaMemcpy(dA, A.data(), A.size() * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dB, B.data(), B.size() * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dAr, Ar.data(), Ar.size() * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dBr, Br.data(), Br.size() * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dA3, A3.data(), A3.size() * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dB3, B3.data(), B3.size() * 4, cudaMemcpyHostToDevice));
  const int smem = 2 * 49152 + 2 * 12800 + 9216 + 8192;
  CK(cudaFuncSetAttribute(umma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  umma_kernel<<<1, 128, smem>>>(dA, dB, dAr, dBr, dA3, dB3, dout, test, argc > 2 ? atoi(argv[2]) : 0);
  printf("test %d\n", test);
  CK(cudaDeviceSynchronize());
  std::vector<char> hb(sizeof(Out));
  CK(cudaMemcpy(hb.data(), dout, sizeof(Out), cudaMemcpyDeviceToHost));
  Out* o = reinterpret_cast<Out*>(hb.data());
  // T1/T2
  double e1 = 0, e2 = 0;
  for (int m = 0; m < 128; ++m)
    for (int n = 0; n < 32; ++n) {
      double r = 0;
      for (int k = 0; k < 96; ++k) r += (double)A[m * 96 + k] * B[n * 96 + k];
      e1 = fmax(e1, fabs(o->d1[m * 32 + n] - r));
      e2 = fmax(e2, fabs(o->d2[m * 32 + n] - r));
    }
  printf("T1 SS exact: max abs err %.3g  (d1[0]=%g d1[33]=%g)\n", e1, o->d1[0], o->d1[33]);
  printf("T2 TS exact: max abs err %.3g\n", e2);
  // T3: with the shared start, row m of every MMA reads smem rows m of sA3 = net (m/32) row m%32 -> D3 region q, lane m
  // holds sum_k A3[m/32][m%32][k] * B3[n][k] for every q. The useful lanes for net q are 32q..32q+31 of region q.
  double e3 = 0;
  for (int m = 0; m < 96; ++m)
    for (int n = 0; n < 32; ++n) {
      const int region = n / 16, nn = n % 16;
      (void)region;
      double r = 0;
      for (int k = 0; k < 24; ++k) r += (double)A3[(m / 32) * 32 * 24 + (m % 32) * 24 + k] * B3[nn * 24 + k];
      e3 = fmax(e3, fabs(o->d3[m * 32 + n] - r));
    }
  printf("T3 stacked-rows (lanes 0..95, regions 0,1): max abs err %.3g\n", e3);
  // T4
  double e4 = 0, e4t = 0, ref_max = 0;
  for (int m = 0; m < 128; ++m)
    for (int n = 0; n < 32; ++n) {
      double r = 0, rt = 0;
      for (int k = 0; k < 96; ++k) {
        r += (double)Ar[m * 96 + k] * Br[n * 96 + k];
        rt += (double)tf32_rna(Ar[m * 96 + k]) * tf32_rna(Br[n * 96 + k]);
      }
      e4 = fmax(e4, fabs(o->d4[m * 32 + n] - r));
      e4t = fmax(e4t, fabs(rt - r));
      ref_max = fmax(ref_max, fabs(r));
    }
  printf("T4 3xTF32: max abs err %.3g (1xTF32 would be %.3g), max |ref| %.3g -> rel %.3g\n", e4, e4t, ref_max, e4 / ref_max);
  if (test == 7) {
    printf("T7 probe (byte offsets of B(n,k), LBO=2048 SBO=512): rows k=0..7, cols n=0..15\n");
    for (int m = 0; m < 8; ++m) {
      for (int n = 0; n < 16; ++n) printf("%6d", (int)(o->d1[m * 32 + n] * 4));
      printf("\n");
    }
  }
  if (test == 8) {
    // D[m][n] = word index of B(n, k=m); expected byte(n, k) = (n/8)*128 + (n%8)*16 + (k/4)*784 + (k%4)*4
    int bad = 0;
    printf("T8 probe (byte offsets of B(n,k), N=48, LBO=784 SBO=128): rows k=0..7, cols n=0..47\n");
    for (int m = 0; m < 8; ++m) {
      for (int n = 0; n < 48; ++n) {
        const int got = (int)((n < 32 ? o->d1[m * 32 + n] : o->d2[m * 32 + n - 32]) * 4);
        bad += got != (int)kmaj_off(n, m, B_SBO, b_lbo(48));
        printf("%5d", got);
      }
      printf("\n");
    }
    printf("T8 N=48 layout: %d of 384 offsets differ from (n/8)*128 + (n%%8)*16 + (k/4)*784 + (k%%4)*4\n", bad);
  }
  if (test == 6) {
    double e6 = 0;
    for (int m = 0; m < 128; ++m)
      for (int n = 0; n < 16; ++n) {
        double r = 0;
        for (int kk = 0; kk < 56; ++kk) r += (double)A[m * 96 + kk] * B[n * 96 + ((50 + kk) % 96)];
        e6 = fmax(e6, fabs(o->d1[m * 32 + n] - r));
      }
    printf("T6 TS + MN-major B window: max abs err %.3g\n", e6);
  }
  printf("T5 cycles total(issue-only): 72 SS N32 %lld(%lld) | 72 TS N32 %lld(%lld) | 72 SS N16 %lld(%lld) | 72 TS N16 %lld(%lld) | 144 TS N16 %lld(%lld) | 144 TS N32 %lld(%lld) | 144 TS N48 %lld(%lld) | 144 TS N64 %lld(%lld) | 1 MMA rt %lld | ld.x32 %lld\n",
         o->t[1], o->t[17], o->t[2], o->t[18], o->t[3], o->t[19], o->t[4], o->t[20], o->t[5], o->t[21], o->t[6], o->t[22], o->t[9], o->t[25], o->t[7], o->t[23], o->t[0], o->t[8]);
  if (test == 5)
    printf("T5 cycles per TS MMA (144 back to back): N16 %.1f | N32 %.1f | N48 %.1f | N64 %.1f\n", o->t[5] / 144.0, o->t[6] / 144.0, o->t[9] / 144.0, o->t[7] / 144.0);
  return 0;
}
