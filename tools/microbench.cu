// microbench.cu -- design-constant measurements for the fused WaveNet kernel (sm_100a).
//   1. FP32 FMA issue rate: scalar FFMA vs packed FFMA2, by resident warps per SM
//   2. the kernel's inner-loop pattern: one warp-uniform weight row (16 floats = 4 x LDS.128)
//      feeding S x 8 FFMA2 (S = time steps per thread); weights from shared memory or from
//      __constant__ memory
//   3. `microbench packed-const`: the compiled kernel's pattern, packed FFMA2 with constant-bank weight pairs
//      against FFMA-immediate
// Prints one JSON object per line.  Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o microbench microbench.cu
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <string>
#include <utility>
#include <vector>

#define CK(x)                                                                                                        \
  do                                                                                                                 \
  {                                                                                                                  \
    cudaError_t e = (x);                                                                                             \
    if (e != cudaSuccess)                                                                                            \
    {                                                                                                                \
      fprintf(stderr, "%s: %s\n", #x, cudaGetErrorString(e));                                                        \
      exit(1);                                                                                                       \
    }                                                                                                                \
  } while (0)

template <bool PACKED>
__global__ void fma_peak(float* out, int iters, float seed)
{
  float2 a[8];
#pragma unroll
  for (int i = 0; i < 8; i++)
    a[i] = make_float2(seed + i, seed - i);
  const float2 m = make_float2(1.0000001f, 0.9999999f);
  const float2 c = make_float2(1e-7f, -1e-7f);
  for (int it = 0; it < iters; it++)
  {
#pragma unroll
    for (int i = 0; i < 8; i++)
    {
      if (PACKED)
        a[i] = __ffma2_rn(a[i], m, c);
      else
      {
        a[i].x = fmaf(a[i].x, m.x, c.x);
        a[i].y = fmaf(a[i].y, m.y, c.y);
      }
    }
  }
  float s = 0.0f;
#pragma unroll
  for (int i = 0; i < 8; i++)
    s += a[i].x + a[i].y;
  if (s == 12345.678f)
    out[0] = s;
}

constexpr int kRows = 1024; // weight rows of 16 floats in the shared-memory variant (64 KB)
constexpr int kConstRows = 896; // 896 rows x 16 floats = 56 KB: the size of the a1_standard weight blob
__constant__ float4 c_weights[kConstRows * 4];

// S time steps per thread, 16 output channels (8 float2 accumulators per time step)
// TAPS: every 4 rows (one plane of 4 input channels) each thread also fetches its S input vectors with
// per-lane LDS.128 (4 wavefronts each), like the real kernel's dilated-tap reads.
template <int S, bool FROM_CONST, bool TAPS>
__global__ void __launch_bounds__(128) inner_loop(const float4* __restrict__ w, float* out, int rows, int iters)
{
  extern __shared__ float4 sw[];
  __shared__ float4 taps[4 * 160];
  if (!FROM_CONST)
  {
    for (int i = threadIdx.x; i < rows * 4; i += blockDim.x)
      sw[i] = w[i];
  }
  for (int i = threadIdx.x; i < 4 * 160; i += blockDim.x)
    taps[i] = make_float4(1e-3f * i, 2e-3f * i, -1e-3f * i, 1e-4f * i);
  __syncthreads();
  float2 acc[S][8];
  float x[S];
#pragma unroll
  for (int j = 0; j < S; j++)
  {
    x[j] = 0.001f * (threadIdx.x + j);
#pragma unroll
    for (int q = 0; q < 8; q++)
      acc[j][q] = make_float2(0.f, 0.f);
  }
  for (int it = 0; it < iters; it++)
  {
#pragma unroll 4
    for (int r = 0; r < rows; r++)
    {
      if (TAPS && (r & 3) == 0)
      {
#pragma unroll
        for (int j = 0; j < S; j++)
        {
          const float4 t = taps[((r >> 2) & 3) * 160 + ((threadIdx.x + 8 * j + it) & 127)];
          x[j] = t.x + t.y + t.z + t.w;
        }
      }
      float4 wq[4];
#pragma unroll
      for (int q = 0; q < 4; q++)
        wq[q] = FROM_CONST ? c_weights[r * 4 + q] : sw[r * 4 + q];
#pragma unroll
      for (int j = 0; j < S; j++)
      {
        const float2 xx = make_float2(x[j], x[j]);
#pragma unroll
        for (int q = 0; q < 4; q++)
        {
          acc[j][2 * q] = __ffma2_rn(make_float2(wq[q].x, wq[q].y), xx, acc[j][2 * q]);
          acc[j][2 * q + 1] = __ffma2_rn(make_float2(wq[q].z, wq[q].w), xx, acc[j][2 * q + 1]);
        }
        x[j] += 1e-6f;
      }
    }
  }
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < S; j++)
#pragma unroll
    for (int q = 0; q < 8; q++)
      s += acc[j][q].x + acc[j][q].y;
  if (s == 12345.678f)
    out[0] = s;
}

// 3. The compiled kernel's straight-line pattern at one frame per thread, 16 channels, over a weight image the size
// of a1_standard's (c_weights: 896 rows of 16 floats = 56 KB), layers of 16 rows whose outputs feed the next layer's
// inputs.
//   PACKED = false: scalar FFMA with the weight as immediate (what wavenet_spec_kernel compiles to today).
//   PACKED = true:  FFMA2 over output-channel pairs, input broadcast from one register, the weight pair from a uniform
//                   register loaded from the constant bank (LDCU.128 = two pairs per load).
constexpr int kPackedConstRows = kConstRows;

__host__ __device__ constexpr float packed_const_weight(int r, int o)
{
  return 0.0625f + 1e-3f * ((r * 16 + o) % 97);
}

// One layer: 16 rows at compile-time offsets (every weight an immediate or a constant-bank address), then its outputs
// become the next layer's inputs.
template <bool PACKED, int L>
__device__ __forceinline__ void packed_const_layer(float (&x)[16], float2 (&acc)[8])
{
#pragma unroll
  for (int i = 0; i < 16; i++)
  {
    const int r = L * 16 + i;
    if (PACKED)
    {
      const float2 xx = make_float2(x[i], x[i]);
#pragma unroll
      for (int q = 0; q < 4; q++)
      {
        const float4 w = c_weights[r * 4 + q];
        acc[2 * q] = __ffma2_rn(xx, make_float2(w.x, w.y), acc[2 * q]);
        acc[2 * q + 1] = __ffma2_rn(xx, make_float2(w.z, w.w), acc[2 * q + 1]);
      }
    }
    else
    {
#pragma unroll
      for (int q = 0; q < 8; q++)
      {
        acc[q].x = fmaf(x[i], packed_const_weight(r, 2 * q), acc[q].x);
        acc[q].y = fmaf(x[i], packed_const_weight(r, 2 * q + 1), acc[q].y);
      }
    }
  }
#pragma unroll
  for (int q = 0; q < 8; q++)
  {
    x[2 * q] = acc[q].x;
    x[2 * q + 1] = acc[q].y;
  }
}

template <bool PACKED, int... L>
__device__ __forceinline__ void packed_const_layers(float (&x)[16], float2 (&acc)[8], std::integer_sequence<int, L...>)
{
  (packed_const_layer<PACKED, L>(x, acc), ...);
}

template <bool PACKED, int MIN_CTAS>
__global__ void __launch_bounds__(512, MIN_CTAS) packed_const(float* out, long long* cycles, int iters)
{
  float x[16];
  float2 acc[8];
#pragma unroll
  for (int i = 0; i < 16; i++)
    x[i] = 1e-3f * (threadIdx.x + i);
#pragma unroll
  for (int q = 0; q < 8; q++)
    acc[q] = make_float2(0.f, 0.f);
  const long long t0 = clock64();
  for (int it = 0; it < iters; it++)
    packed_const_layers<PACKED>(x, acc, std::make_integer_sequence<int, kPackedConstRows / 16>{});
  if (threadIdx.x == 0 && blockIdx.x == 0)
    cycles[0] = clock64() - t0;
  float s = 0.f;
#pragma unroll
  for (int q = 0; q < 8; q++)
    s += acc[q].x + acc[q].y;
  if (s == 12345.678f)
    out[0] = s;
}

static double time_ms(cudaEvent_t e0, cudaEvent_t e1)
{
  float ms;
  CK(cudaEventSynchronize(e1));
  CK(cudaEventElapsedTime(&ms, e0, e1));
  return ms;
}

// `microbench packed-const`: FMA/clk/SM of the packed constant-bank form against scalar FFMA-immediate, 16/32/64
// warps per SM, 512-thread CTAs, one wave.  Per clock is given both at the attribute's max clock (comparable with the
// other tests) and at the SM clock block 0 counted during the run.
static void run_packed_const(int sms, int clock_khz, float* d, cudaEvent_t e0, cudaEvent_t e1)
{
  std::vector<float4> hw(kPackedConstRows * 4);
  for (int r = 0; r < kPackedConstRows; r++)
    for (int q = 0; q < 4; q++)
      hw[r * 4 + q] = make_float4(packed_const_weight(r, 4 * q), packed_const_weight(r, 4 * q + 1),
                                  packed_const_weight(r, 4 * q + 2),
                                  packed_const_weight(r, 4 * q + 3));
  CK(cudaMemcpyToSymbol(c_weights, hw.data(), sizeof(float4) * hw.size()));
  long long* dcyc;
  CK(cudaMalloc(&dcyc, sizeof(long long)));
  const int iters = 256;
  for (int warps_per_sm : {16, 32, 64})
    for (int packed = 0; packed < 2; packed++)
    {
      const int ctas_per_sm = warps_per_sm / 16, blocks = sms * ctas_per_sm;
      auto kern = packed ? (warps_per_sm == 64 ? packed_const<true, 4> : packed_const<true, 2>)
                         : (warps_per_sm == 64 ? packed_const<false, 4> : packed_const<false, 2>);
      cudaFuncAttributes fa;
      CK(cudaFuncGetAttributes(&fa, kern));
      double best = 1e30;
      long long cyc = 0, hcyc = 0;
      for (int rep = 0; rep < 5; rep++) // rep 0 warms up
      {
        CK(cudaEventRecord(e0));
        kern<<<blocks, 512>>>(d, dcyc, iters);
        CK(cudaEventRecord(e1));
        const double ms = time_ms(e0, e1);
        CK(cudaMemcpy(&hcyc, dcyc, sizeof(hcyc), cudaMemcpyDeviceToHost));
        if (rep > 0 && ms < best)
        {
          best = ms;
          cyc = hcyc;
        }
      }
      const double fma_per_sm = 16.0 * kPackedConstRows * iters * 512.0 * ctas_per_sm;
      printf("{\"test\": \"packed_const\", \"form\": \"%s\", \"warps_per_sm\": %d, \"ms\": %.3f, "
             "\"sm_clock_mhz\": %.0f, \"fma_per_clk_per_sm_at_max_clock\": %.1f, \"fma_per_clk_per_sm\": %.1f, "
             "\"regs\": %d, \"spill_bytes\": %d}\n",
             packed ? "FFMA2 x-broadcast, UR weight pair (LDCU.128)" : "FFMA immediate", warps_per_sm, best,
             cyc / (best * 1e3), fma_per_sm / (best * 1e-3) / (clock_khz * 1e3), fma_per_sm / cyc, fa.numRegs,
             (int)fa.localSizeBytes);
    }
  CK(cudaFree(dcyc));
}

int main(int argc, char** argv)
{
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, 0));
  const int sms = prop.multiProcessorCount;
  int clock_khz = 0;
  CK(cudaDeviceGetAttribute(&clock_khz, cudaDevAttrClockRate, 0));
  printf("{\"device\": \"%s\", \"sms\": %d, \"max_clock_mhz\": %d}\n", prop.name, sms, clock_khz / 1000);
  float* d;
  CK(cudaMalloc(&d, 4));
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0));
  CK(cudaEventCreate(&e1));
  if (argc > 1 && std::string(argv[1]) == "packed-const")
  {
    run_packed_const(sms, clock_khz, d, e0, e1);
    return 0;
  }

  // 1. raw FMA peaks vs resident warps per SM
  for (int packed = 0; packed < 2; packed++)
    for (int warps_per_sm : {4, 8, 16, 32, 64})
    {
      const int threads = 128, blocks = sms * (warps_per_sm / 4), iters = 8192;
      double best = 1e30;
      for (int rep = 0; rep < 4; rep++)
      {
        CK(cudaEventRecord(e0));
        if (packed)
          fma_peak<true><<<blocks, threads>>>(d, iters, 1.f);
        else
          fma_peak<false><<<blocks, threads>>>(d, iters, 1.f);
        CK(cudaEventRecord(e1));
        best = fmin(best, time_ms(e0, e1));
      }
      const double fma = 16.0 * iters * (double)blocks * threads;
      printf("{\"test\": \"fma_peak\", \"packed\": %d, \"warps_per_sm\": %d, \"tflops\": %.2f, \"fma_per_clk_per_sm_at_max_clock\": %.1f}\n",
             packed, warps_per_sm, 2 * fma / (best * 1e-3) / 1e12, fma / (best * 1e-3) / sms / (clock_khz * 1e3));
    }

  // 2. inner loop pattern
  std::vector<float4> hw(kRows * 4);
  for (size_t i = 0; i < hw.size(); i++)
    hw[i] = make_float4(1e-3f * (i % 7), -1e-3f * (i % 5), 1e-3f, -1e-3f);
  float4* dw;
  CK(cudaMalloc(&dw, hw.size() * sizeof(float4)));
  CK(cudaMemcpy(dw, hw.data(), hw.size() * sizeof(float4), cudaMemcpyHostToDevice));
  CK(cudaMemcpyToSymbol(c_weights, hw.data(), sizeof(float4) * kConstRows * 4));
  const int iters = 64;
  const size_t smem = kRows * 4 * sizeof(float4); // 64 KB
#define RUN_INNER(SVAL, CONSTV, TAPSV)                                                                               \
  for (int ctas_per_sm : {1, 2, 3, 4})                                                                               \
  {                                                                                                                  \
    const int rows = CONSTV ? kConstRows : kRows;                                                                    \
    auto kern = inner_loop<SVAL, CONSTV, TAPSV>;                                                                     \
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                          \
    const int blocks = sms * ctas_per_sm;                                                                            \
    double best = 1e30;                                                                                              \
    for (int rep = 0; rep < 4; rep++)                                                                                \
    {                                                                                                                \
      CK(cudaEventRecord(e0));                                                                                       \
      kern<<<blocks, 128, CONSTV ? 0 : smem>>>(dw, d, rows, iters);                                                  \
      CK(cudaEventRecord(e1));                                                                                       \
      best = fmin(best, time_ms(e0, e1));                                                                            \
    }                                                                                                                \
    const double fma = 16.0 * SVAL * rows * (double)iters * blocks * 128;                                            \
    printf("{\"test\": \"inner_loop\", \"S\": %d, \"weights\": \"%s\", \"taps\": %d, \"ctas_per_sm\": %d, \"tflops\": %.2f, " \
           "\"fma_per_clk_per_sm_at_max_clock\": %.1f}\n",                                                           \
           SVAL, CONSTV ? "constant" : "shared", (int)TAPSV, ctas_per_sm, 2 * fma / (best * 1e-3) / 1e12,            \
           fma / (best * 1e-3) / sms / (clock_khz * 1e3));                                                           \
  }
  RUN_INNER(2, false, false)
  RUN_INNER(2, false, true)
  RUN_INNER(4, false, true)
  RUN_INNER(2, true, false)
  RUN_INNER(2, true, true)
  RUN_INNER(4, true, true)
  return 0;
}
