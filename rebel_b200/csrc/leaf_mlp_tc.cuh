// Primitives and the weight-blob layout of the tcgen05 value net (the kernel: leaf_mlp_tc3.cuh).  The net is Net2: Linear ->
// LayerNorm -> GELU -> Linear -> LayerNorm -> GELU -> Linear (cfvpy/models.py:64-94), evaluated with tcgen05.mma (kind::f16, fp16
// operands, fp32 accumulation in TMEM) on 128-row tiles of pseudo-leaf query rows.
//
// Shapes shared by the host and the kernel: 544 threads per CTA, warps 0-15 = epilogue (warp w owns TMEM lanes 32*(w&3).., one
// row per thread, and the column quarter (w>>2) of the 256 hidden features), warp 16 = TMEM allocator + single-thread MMA issuer.
// The biases ride on the tensor cores: layer 1 through a constant-1 query column (written by the CFR kernel) against a bias
// column in W1, layer 2 through one extra K=16 MMA of a constant "ones" tile against a bias tile; both live in the blob.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace cfrb {
namespace tc {

constexpr int kHid = 256;
constexpr int kTileM = 128;
constexpr int kNout = 16;                 // output features padded to the minimum UMMA N
constexpr int kParts = 4;                    // column quarters per row
constexpr int kColsPerThread = kHid / kParts;   // 64
constexpr int kEpiThreads = 128 * kParts;    // 16 epilogue warps
constexpr int kSubChunks = 4;                // A-operand hand-over granularity: 16 features per thread
constexpr int kThreads = kEpiThreads + 32;   // + allocator / MMA-issuer warp
constexpr uint32_t kColD = 0, kTmemCols = 512;

// ---- weight-blob layout (bytes).  The blob in global memory has exactly the shared-memory layout up to off_x.
struct BlobLayout {
  int Kp;            // padded query width (multiple of 16, with at least one spare column for the constant 1)
  int off_w1, off_w2, off_w3, off_ones, off_bias2, off_ln1, off_ln2, off_b3, blob_bytes, off_x;
  __host__ __device__ explicit BlobLayout(int kp) : Kp(kp) {
    off_w1 = 0;                               // [256 x Kp]  fp16, column Q holds bias 1
    off_w2 = off_w1 + kHid * kp * 2;          // [256 x 256] fp16
    off_w3 = off_w2 + kHid * kHid * 2;        // [16 x 256]  fp16
    off_ones = off_w3 + kNout * kHid * 2;     // [128 x 16]  fp16, column 0 = 1
    off_bias2 = off_ones + kTileM * 16 * 2;   // [256 x 16]  fp16, column 0 = bias 2
    off_ln1 = off_bias2 + kHid * 16 * 2;      // float4 {gamma_j, gamma_j+1, beta_j, beta_j+1} per feature pair
    off_ln2 = off_ln1 + kHid * 8;
    off_b3 = off_ln2 + kHid * 8;
    blob_bytes = off_b3 + kNout * 4;
    off_x = (blob_bytes + 127) / 128 * 128;   // first byte of shared memory after the weights (Tc3Layout)
  }
};

// Element (row r, col k) of a K-major [R x K] fp16 operand in UMMA "no swizzle" core-matrix order:
// 8x8 core matrices of 128 contiguous bytes; row-groups are 128 B apart (SBO), K-chunks R/8*128 B apart (LBO).
__host__ __device__ inline int umma_kmajor_offset_halves(int r, int k, int R) {
  return (k >> 3) * (R >> 3) * 64 + (r >> 3) * 64 + (r & 7) * 8 + (k & 7);
}

// ---------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra WAIT_DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc),
      "r"(accumulate) : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem desc]
__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc),
      "r"(accumulate) : "memory");
}
// UMMA shared-memory descriptor, K-major, SWIZZLE_NONE (cute::UMMA::SmemDescriptor): start>>4 [0,14), LBO>>4 [16,30),
// SBO>>4 [32,46), version=1 [46,48), layout_type=0 [61,64).
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) |
         (1ull << 46);
}
// Instruction descriptor (cute::UMMA::InstrDescriptor): D=f32 [4,6)=1, A/B format f16=0 [7,10),[10,13), both K-major,
// N>>3 at [17,23), M>>4 at [24,29).
__device__ __forceinline__ constexpr uint32_t make_idesc(int M, int N) {
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

#define CFRB_TMEM_LD32(taddr, v)                                                                                          \
  asm volatile(                                                                                                           \
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "                                                                           \
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, " \
      "[%32];"                                                                                                            \
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),      \
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),            \
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),           \
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])                         \
      : "r"(taddr))

#define CFRB_TMEM_LD16(taddr, v)                                                                                          \
  asm volatile(                                                                                                           \
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"           \
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),      \
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])                          \
      : "r"(taddr))

#define CFRB_TMEM_ST8(taddr, v)                                                                                           \
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(v[0]), "r"(v[1]),  \
               "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])                                           \
               : "memory")

__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// Packed fp32 pairs (Blackwell FFMA2 / FADD2): one issue slot for two lanes' worth of LayerNorm arithmetic.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
  f32x2 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}

// GELU(y) = y * Phi(y), Phi(y) = 0.5 (1 + erf(y / sqrt 2)).  erf(z) = tanh(z (a + b z^2 + c z^4)) to 1.0e-4 (fitted, max error
// of the resulting GELU 2.5e-5 absolute — 20x below the fp16 rounding of the activation it feeds), evaluated as a logistic
// with ex2 / rcp so it is branch-free: y / (1 + 2^(-2 log2(e) u)), u = y (c0 + c1 y^2 + c2 y^4).
__device__ __forceinline__ float gelu_tc(float y) {
  const float y2 = fminf(y * y, 52.f);                              // beyond |y| ~ 7.2 the logistic is saturated anyway
  // -2 log2(e) * (c0 + c1 y^2 + c2 y^4)
  const float p = fmaf(y2, fmaf(y2, 1.014244e-3f, -1.0677588e-1f), -2.3011216f);
  const float t = y * p;
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(t));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
  return y * r;
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

struct TcArgs {
  const uint8_t* blob;      // weights in smem layout (BlobLayout)
  const __half* Xh;         // [tiles][Kp/8][16][8][8] fp16 query tiles
  const int* rows_ptr;
  float* out;               // [rows][Hout]
  int Kp, H, Hout;
  float* dbg_d1;            // optional [128][256] raw layer-1 accumulators of tile 0
  float* dbg_d2;            // optional [128][256] raw layer-2 accumulators of tile 0
  long long* trace;         // optional (debug launch only): SM clock stamps of CTA 0, [2048]: epilogue thread 0 at
                            // [phase*8 + e], MMA issuer at [1024 + phase*4 + m]
};

}  // namespace tc
}  // namespace cfrb
