// CFR wave kernels, compiled as their own translation unit with -fmad=false: without fused multiply-adds every fp64
// operation is an individually rounded IEEE operation in the same order as the reference's scalar C++ (built without
// contraction), which makes the CFRB_STATE_F64 path reproduce the reference bit for bit between value-net calls.
#include <algorithm>

#include "cfr_kernels.cuh"
#include "br_kernel.cuh"
#include "selfplay_kernels.cuh"

namespace cfrb {

// Hand counts with a compile-time specialisation (1x4f, 1x5f, 1x6f, 2x3f, 2x4f); anything else takes the generic path.
#define CFRB_DISPATCH_H(H, CALL)          \
  switch (H) {                            \
    case 4: { CALL(4); break; }           \
    case 5: { CALL(5); break; }           \
    case 6: { CALL(6); break; }           \
    case 9: { CALL(9); break; }           \
    case 16: { CALL(16); break; }         \
    default: { CALL(0); break; }          \
  }

template <typename real>
cudaError_t cfr_configure(int group, int smem_bytes) {
  if (group != 32) return cudaSuccess;
  cudaError_t e = cudaSuccess;
#define CFRB_CFG(HC)                                                                                                      \
  if (e == cudaSuccess) e = cudaFuncSetAttribute(cfr_iter_kernel<real, 32, HC>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
  CFRB_CFG(0) CFRB_CFG(4) CFRB_CFG(5) CFRB_CFG(6) CFRB_CFG(9) CFRB_CFG(16)
#undef CFRB_CFG
  if (e != cudaSuccess) return e;
  return cudaFuncSetAttribute(cfr_init_kernel<real, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
}

template <typename real>
void cfr_launch_init(const CfrDev<real>& p, int group, int blocks, int threads, size_t smem, cudaStream_t st, int scratch_per_group) {
  if (group == 32) cfr_init_kernel<real, 32><<<blocks, threads, smem, st>>>(p, scratch_per_group);
  else cfr_init_kernel<real, 256><<<blocks, 256, 0, st>>>(p, scratch_per_group);
}

template <typename real>
void cfr_launch_iter(const CfrDev<real>& p, int group, int blocks, int threads, size_t smem, cudaStream_t st, int iter, int do_b,
                     int do_f, int scratch_per_group) {
  if (group == 32) {
#define CFRB_CALL(HC) cfr_iter_kernel<real, 32, HC><<<blocks, threads, smem, st>>>(p, iter, do_b, do_f, scratch_per_group)
    CFRB_DISPATCH_H(p.H, CFRB_CALL)
#undef CFRB_CALL
  } else {
    cfr_iter_kernel<real, 256, 0><<<blocks, 256, 0, st>>>(p, iter, do_b, do_f, scratch_per_group);
  }
}

void br_launch(const BrDev& p, cudaStream_t st) { br_kernel<<<2, 1024, 0, st>>>(p); }

template <typename real>
cudaError_t cfr_configure_d2(int smem_bytes) {
  cudaError_t e = cudaSuccess;
#define CFRB_CFG(HC)                                                                                                      \
  if (e == cudaSuccess) e = cudaFuncSetAttribute(cfr_iter_d2_kernel<real, HC>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
  CFRB_CFG(0) CFRB_CFG(4) CFRB_CFG(5) CFRB_CFG(6) CFRB_CFG(9) CFRB_CFG(16)
#undef CFRB_CFG
  return e;
}

// Launch with programmatic stream serialization (PDL): the grid may start before its predecessor in the stream has finished;
// the kernel orders itself with griddepcontrol.wait.  Captured into CUDA graphs as a programmatic dependency edge.
template <typename... KArgs, typename... Args>
static void launch_pdl(void (*kernel)(KArgs...), int blocks, int threads, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(blocks); cfg.blockDim = dim3(threads); cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, kernel, args...);
}

template <typename real>
void cfr_launch_iter_d2(const CfrDev<real>& p, int blocks, int threads, size_t smem, cudaStream_t st, int iter, int do_b, int do_f,
                        int scratch_per_group) {
#define CFRB_CALL(HC) launch_pdl(cfr_iter_d2_kernel<real, HC>, blocks, threads, smem, st, p, iter, do_b, do_f, scratch_per_group)
  CFRB_DISPATCH_H(p.H, CFRB_CALL)
#undef CFRB_CALL
}

void sp_launch_seed(const SpDev& p, const uint32_t* dev_seeds, cudaStream_t st) {
  sp_seed_kernel<<<(p.K + 127) / 128, 128, 0, st>>>(p, dev_seeds);
}
template <typename real>
void sp_launch_begin(const SpDev& p, real* wave_beliefs, cudaStream_t st) {
  sp_begin_kernel<real><<<(p.K + 127) / 128, 128, 0, st>>>(p, wave_beliefs);
  sp_scan_kernel<<<1, 1024, 0, st>>>(p);
}
template <typename real>
void sp_launch_finish(const SpDev& p, const real* mu, const real* snap, float* ex_q, float* ex_v, cudaStream_t st) {
  if (ex_q) sp_examples_kernel<real><<<(2 * p.K + 127) / 128, 128, 0, st>>>(p, mu, ex_q, ex_v);
  sp_advance_kernel<real><<<(p.K + 127) / 128, 128, 0, st>>>(p, snap);
}
__global__ void rows_gather_kernel(const float* __restrict__ src, int width, const int* __restrict__ ids, int n, float* __restrict__ out) {
  const size_t total = (size_t)n * width;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / width), c = (int)(i % width);
    out[i] = src[(size_t)ids[r] * width + c];
  }
}
void rows_launch_gather(const float* src, int width, const int* ids, int n, float* out, cudaStream_t st) {
  if (n <= 0) return;
  const size_t total = (size_t)n * width;
  const int blocks = (int)std::min<size_t>((total + 255) / 256, 148 * 8);
  rows_gather_kernel<<<blocks, 256, 0, st>>>(src, width, ids, n, out);
}

// div_by_rcp against IEEE division on pseudo-random operands: quotient mantissas spread over [1, 2), including operands whose
// quotient lies within a few ulp of a power of two and denominators with all-ones / all-zeros low mantissa bits.
__global__ void div_check_kernel(unsigned long long seed, unsigned long long* mismatches) {
  unsigned long long s = seed + (unsigned long long)(blockIdx.x * blockDim.x + threadIdx.x) * 0x9E3779B97F4A7C15ull;
  auto next = [&]() { s ^= s << 13; s ^= s >> 7; s ^= s << 17; return s; };
  unsigned long long bad = 0;
  for (int i = 0; i < 4096; ++i) {
    const unsigned long long a = next(), c = next(), m = next();
    double b = __longlong_as_double((long long)(0x3FF0000000000000ull | (c >> 12)));           // [1, 2)
    double x = __longlong_as_double((long long)(0x3FF0000000000000ull | (a >> 12)));
    const int kind = (int)(m & 7);
    if (kind == 1) b = __longlong_as_double((long long)(0x3FFFFFFFFFFFFF00ull | (c & 0xFF)));     // denominator just below 2
    if (kind == 2) b = __longlong_as_double((long long)(0x3FF0000000000000ull | (c & 0xFF)));     // just above 1
    if (kind == 3) x = b * (1.0 + (double)((long long)(a & 0xF) - 8) * 2.220446049250313e-16);      // quotient within a few ulp of 1
    if (kind == 4) x = x * 1e-80;                                                                   // the smoothing epsilon's scale
    if (kind == 5) b = b * (double)(1 + (c & 15));                                                  // sums of up to a dozen regrets
    const double y = 1.0 / b;
    const double q = div_by_rcp(x, b, y);
    if (__double_as_longlong(q) != __double_as_longlong(x / b)) ++bad;
  }
  if (bad) atomicAdd(mismatches, bad);
}
void div_check_launch(unsigned long long seed, int blocks, unsigned long long* mismatches, cudaStream_t st) {
  div_check_kernel<<<blocks, 256, 0, st>>>(seed, mismatches);
}

#define CFRB_INSTANTIATE(real)                                                                                             \
  template cudaError_t cfr_configure<real>(int, int);                                                                      \
  template void cfr_launch_init<real>(const CfrDev<real>&, int, int, int, size_t, cudaStream_t, int);                      \
  template void cfr_launch_iter<real>(const CfrDev<real>&, int, int, int, size_t, cudaStream_t, int, int, int, int);             \
  template cudaError_t cfr_configure_d2<real>(int);                                                                        \
  template void cfr_launch_iter_d2<real>(const CfrDev<real>&, int, int, size_t, cudaStream_t, int, int, int, int);                \
  template void sp_launch_begin<real>(const SpDev&, real*, cudaStream_t);                                                  \
  template void sp_launch_finish<real>(const SpDev&, const real*, const real*, float*, float*, cudaStream_t);
CFRB_INSTANTIATE(float)
CFRB_INSTANTIATE(double)

}  // namespace cfrb
