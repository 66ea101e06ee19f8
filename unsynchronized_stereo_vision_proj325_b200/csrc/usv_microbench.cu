// usv_microbench.cu — register-only issue-rate probes for the packed-byte integer
// instructions the block-search kernels are built from (SURVEY.md 8(d): the ALU
// roofline denominator is not in MEASURED_PEAKS.json and must be measured).
// Prints one JSON line per probe: lanes/clk/SM derived from clock64() inside the
// kernel (independent of the boost clock) and G inst/s from CUDA events.
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o usv_microbench usv_microbench.cu
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <vector>

#define CK(x)                                                                              \
  do {                                                                                     \
    cudaError_t e = (x);                                                                   \
    if (e != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e), __FILE__, __LINE__); exit(1); } \
  } while (0)

constexpr int kThreads = 256;
constexpr int kIters = 4096;
constexpr int kChains = 8;  // independent dependency chains per thread (ILP)

enum Probe {
  P_SAD4_ACC, P_ABSDIFF4, P_DP4A, P_IADD3, P_IMAD, P_LOP3, P_SHF, P_PRMT, P_VIMNMX, P_LEA,
  P_SAD4_IMAD, P_SAD4_IADD, P_SAD4_VIMNMX, P_DP4A_SAD4, P_DP4A_IMAD, P_SAD4_SHF, P_IADD_IMAD,
  P_SHFL, P_LDS32, P_LDS128, P_SAD4_LDS, P_DMUL, P_SAD4_DMUL, P_REDUX, P_REDUX_STRIDED, P_SAD4_REDUX, P_POPC, P_HAMMING4, P_COUNT
};
static const char* kNames[P_COUNT] = {
  "VABSDIFF4.U8.ACC", "VABSDIFF4.U8", "IDP.4A.U8.U8", "IADD3", "IMAD", "LOP3", "SHF.R.W(funnel)", "PRMT", "VIMNMX.U32", "LEA",
  "VABSDIFF4.ACC+IMAD", "VABSDIFF4.ACC+IADD3", "VABSDIFF4.ACC+VIMNMX", "IDP.4A+VABSDIFF4.ACC", "IDP.4A+IMAD", "VABSDIFF4.ACC+SHF",
  "IADD3+IMAD", "SHFL.BFLY", "LDS.32", "LDS.128", "VABSDIFF4.ACC+LDS.32", "DMUL", "VABSDIFF4.ACC+DMUL",
  "REDUX.MIN.U32(full mask)", "REDUX.MIN.U32(8 lanes, stride 4)", "VABSDIFF4.ACC+REDUX.MIN(stride 4)", "POPC",
  "LOP3+POPC+IADD3(census word)"};
// tested instructions per chain step (for the mixed probes both are counted)
static const int kOpsPerStep[P_COUNT] = {1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 2, 2, 2, 2, 2, 2, 2, 1, 1, 1, 2, 1, 2, 1, 1, 2, 1, 3};

__device__ __forceinline__ uint32_t sad4(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t d;
  asm volatile("vabsdiff4.u32.u32.u32.add %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
__device__ __forceinline__ uint32_t dp4a_u(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t d;
  asm volatile("dp4a.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
__device__ __forceinline__ uint32_t imad(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t d;
  asm volatile("mad.lo.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
__device__ __forceinline__ uint32_t iadd3(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t d;
  asm volatile("{.reg .u32 t; add.u32 t, %1, %2; add.u32 %0, t, %3;}" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
__device__ __forceinline__ uint32_t lop3(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t d;
  asm volatile("lop3.b32 %0, %1, %2, %3, 0x96;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
__device__ __forceinline__ uint32_t popc(uint32_t a) {
  uint32_t d;
  asm volatile("popc.b32 %0, %1;" : "=r"(d) : "r"(a));
  return d;
}
__device__ __forceinline__ uint32_t shf(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t d;
  asm volatile("shf.r.wrap.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t d;
  asm volatile("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
__device__ __forceinline__ uint32_t vmin(uint32_t a, uint32_t b) {
  uint32_t d;
  asm volatile("min.u32 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
  return d;
}
__device__ __forceinline__ uint32_t lea(uint32_t a, uint32_t b) {
  uint32_t d;
  asm volatile("{.reg .u32 t; shl.b32 t, %1, 16; add.u32 %0, t, %2;}" : "=r"(d) : "r"(a), "r"(b));
  return d;
}

template <int P>
__global__ void __launch_bounds__(kThreads) probe_kernel(uint32_t* out, long long* cycles, uint32_t seed_a, uint32_t seed_b) {
  __shared__ uint32_t sm[kThreads * 8];
  uint32_t x[kChains], y[kChains];
  double dx[kChains];
  const uint32_t a = seed_a * (threadIdx.x + 1), b = seed_b + threadIdx.x;
#pragma unroll
  for (int c = 0; c < kChains; ++c) { x[c] = a + c; y[c] = b ^ c; dx[c] = 1.0 + c * 1e-9; }
  for (int i = threadIdx.x; i < kThreads * 8; i += kThreads) sm[i] = i * seed_a;
  __syncthreads();
  const uint32_t* lp = sm + (threadIdx.x * 4) % (kThreads * 4);
  const uint4* lp4 = reinterpret_cast<const uint4*>(sm) + threadIdx.x;
  const double dm = 1.0 + 1e-12 * seed_a;
  long long t0 = clock64();
#pragma unroll 4
  for (int it = 0; it < kIters; ++it) {
#pragma unroll
    for (int c = 0; c < kChains; ++c) {
      if (P == P_SAD4_ACC) x[c] = sad4(a, b, x[c]);
      if (P == P_ABSDIFF4) x[c] = __vabsdiffu4(x[c], b);
      if (P == P_DP4A) x[c] = dp4a_u(a, b, x[c]);
      if (P == P_IADD3) x[c] = iadd3(x[c], a, b);
      if (P == P_IMAD) x[c] = imad(x[c], a, b);
      if (P == P_LOP3) x[c] = lop3(x[c], a, b);
      if (P == P_SHF) x[c] = shf(x[c], a, b);
      if (P == P_PRMT) x[c] = prmt(x[c], a, b);
      if (P == P_VIMNMX) x[c] = vmin(x[c], a);
      if (P == P_LEA) x[c] = lea(x[c], b);
      if (P == P_SAD4_IMAD) { x[c] = sad4(a, b, x[c]); y[c] = imad(y[c], a, b); }
      if (P == P_SAD4_IADD) { x[c] = sad4(a, b, x[c]); y[c] = iadd3(y[c], a, b); }
      if (P == P_SAD4_VIMNMX) { x[c] = sad4(a, b, x[c]); y[c] = vmin(y[c], x[c]); }
      if (P == P_DP4A_SAD4) { x[c] = sad4(a, b, x[c]); y[c] = dp4a_u(a, b, y[c]); }
      if (P == P_DP4A_IMAD) { x[c] = dp4a_u(a, b, x[c]); y[c] = imad(y[c], a, b); }
      if (P == P_SAD4_SHF) { x[c] = sad4(a, b, x[c]); y[c] = shf(y[c], a, b); }
      if (P == P_IADD_IMAD) { x[c] = iadd3(x[c], a, b); y[c] = imad(y[c], a, b); }
      if (P == P_SHFL) x[c] = __shfl_xor_sync(0xffffffffu, x[c], 1);
      if (P == P_LDS32) x[c] += *((volatile const uint32_t*)lp + ((it + c) & 3));
      if (P == P_LDS128) {
        uint4 v;
        unsigned sa = (unsigned)__cvta_generic_to_shared(lp4 + ((it + c) & 1) * kThreads);
        asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(sa));
        x[c] += v.x ^ v.y ^ v.z ^ v.w;
      }
      if (P == P_SAD4_LDS) { x[c] = sad4(a, *((volatile const uint32_t*)lp + ((it + c) & 3)), x[c]); }
      if (P == P_REDUX) x[c] = __reduce_min_sync(0xffffffffu, x[c] + it);
      if (P == P_REDUX_STRIDED) x[c] = __reduce_min_sync(0x11111111u << (threadIdx.x & 3), x[c] + it);
      if (P == P_SAD4_REDUX) { y[c] = sad4(a, b, y[c]); x[c] = __reduce_min_sync(0x11111111u << (threadIdx.x & 3), x[c] + it); }
      if (P == P_POPC) x[c] = popc(x[c]);
      // the census sweep's candidate slot (usv_common.cuh: hamming4_acc): c + popc(a ^ b)
      if (P == P_HAMMING4) x[c] = iadd3(popc(lop3(x[c], a, b)), x[c], a);
      if (P == P_DMUL) dx[c] = __dmul_rn(dx[c], dm);
      if (P == P_SAD4_DMUL) { x[c] = sad4(a, b, x[c]); dx[c] = __dmul_rn(dx[c], dm); }
    }
  }
  long long t1 = clock64();
  uint32_t r = 0;
  double rd = 0;
#pragma unroll
  for (int c = 0; c < kChains; ++c) { r ^= x[c] ^ y[c]; rd += dx[c]; }
  r ^= (uint32_t)__double2loint(rd);
  if (r == seed_b * 0x9e3779b9u) out[0] = r;  // runtime-opaque: keeps the chains alive
  if (threadIdx.x == 0) cycles[blockIdx.x] = t1 - t0;
}

template <int P>
static void run(int sms, int blocks_per_sm, uint32_t* d_out, long long* d_cyc, double* lanes_out) {
  const int grid = sms * blocks_per_sm;
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
  probe_kernel<P><<<grid, kThreads>>>(d_out, d_cyc, 3, 5);  // warm-up
  CK(cudaDeviceSynchronize());
  CK(cudaEventRecord(e0));
  probe_kernel<P><<<grid, kThreads>>>(d_out, d_cyc, 3, 5);
  CK(cudaEventRecord(e1));
  CK(cudaDeviceSynchronize());
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, e0, e1));
  std::vector<long long> cyc(grid);
  CK(cudaMemcpy(cyc.data(), d_cyc, sizeof(long long) * grid, cudaMemcpyDeviceToHost));
  double avg = 0; long long mx = 0;
  for (long long c : cyc) { avg += (double)c; if (c > mx) mx = c; }
  avg /= grid;
  const double inst_per_thread = (double)kIters * kChains * kOpsPerStep[P];
  const double lanes_per_clk_sm = inst_per_thread * kThreads * blocks_per_sm / avg;
  const double ginst = inst_per_thread * kThreads * (double)grid / (ms * 1e-3) / 1e9;
  printf("{\"probe\": \"%s\", \"blocks_per_sm\": %d, \"lanes_per_clk_per_sm\": %.2f, \"gthread_inst_per_s\": %.1f, "
         "\"ms\": %.4f, \"avg_cycles\": %.0f, \"max_cycles\": %lld, \"implied_mhz\": %.0f}\n",
         kNames[P], blocks_per_sm, lanes_per_clk_sm, ginst, ms, avg, mx, avg / (ms * 1e-3) / 1e6);
  if (lanes_out) *lanes_out = lanes_per_clk_sm;
  CK(cudaEventDestroy(e0)); CK(cudaEventDestroy(e1));
}

template <int P>
static void run_all(int sms, uint32_t* d_out, long long* d_cyc) {
  run<P>(sms, 4, d_out, d_cyc, nullptr);
  if constexpr (P + 1 < P_COUNT) run_all<P + 1>(sms, d_out, d_cyc);
}

int main() {
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, 0));
  printf("{\"device\": \"%s\", \"sms\": %d, \"cc\": \"%d.%d\", \"clock_khz\": %d}\n", prop.name, prop.multiProcessorCount, prop.major,
         prop.minor, prop.clockRate);
  uint32_t* d_out; long long* d_cyc;
  CK(cudaMalloc(&d_out, 64));
  CK(cudaMalloc(&d_cyc, sizeof(long long) * prop.multiProcessorCount * 8));
  run_all<0>(prop.multiProcessorCount, d_out, d_cyc);
  // occupancy sweep for the headline instruction
  run<P_SAD4_ACC>(prop.multiProcessorCount, 1, d_out, d_cyc, nullptr);
  run<P_SAD4_ACC>(prop.multiProcessorCount, 2, d_out, d_cyc, nullptr);
  run<P_SAD4_ACC>(prop.multiProcessorCount, 8, d_out, d_cyc, nullptr);
  return 0;
}
