// usv_common.cuh — device-side structs and helpers shared by the sm_100a kernels, and the host pieces the dense sweeps share.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/usv_b200.h"

namespace usv {

// SMs of the device the library runs on (set by usv_create from cudaDeviceProp; B200: 148): grid sizing only
extern int g_sm_count;

// Everything a matching kernel needs, passed by value (fits the 4 KB param space).
struct DevJob {
  const uint8_t* left;
  const uint8_t* right;
  long long frame_stride;
  int width, height, channels, row_stride;
  int tw, th, dmin, dmax, sx, sy;
  int cost_kind, camera_side, distance_kind;
  int nxc, nyc;     // valid window positions per row / column (stride 1)
  int nx, ny;       // window grid
  int row_bytes;    // tw * channels
  int n_elems;      // tw * th * channels
  double accept_threshold;
  // sparse template list (nullptr => dense grid), shared by all pairs
  const int* tx;
  const int* ty;
  int n_templates;  // windows per pair (nx*ny for dense)
  usv_outputs out;
  uint32_t* cost_rows;
  double* score_rows;
  int row_cap;
  const double* dist_lut;  // [width] distance by disparity (dense kernels), may be null
  int corr_kernel;         // USV_CORR_KERNEL_* (usv_set_option): which correlation sweep to run; 0 = automatic
  int* status;             // device-visible status word of the context (mapped host memory): a kernel that gives up
                           // (a tcgen05 wait that exceeds its wall-clock bound) sets it instead of trapping
};

constexpr int kDevStatusUmmaTimeout = 1;

// ---- host side shared by the dense sweeps
// the kernel that serves a matching call (usv_capi.cu: plan_match, whose name tables follow this order; DESIGN §4)
enum class Sweep { kSad, kCensus, kCorrAlu, kCorrMma, kCorrUmma, kDirect, kNone };

// row pitch of the planes that interleaved colour frames are split into for the dense sweeps, and the bytes of the
// planes of one frame (0 for one-plane frames, which are read in place)
inline int colour_plane_pitch(const DevJob& J) { return ((J.width + 15) & ~15) + 16; }
inline size_t colour_planes_bytes(const DevJob& J) { return J.channels > 1 ? (size_t)J.channels * J.height * colour_plane_pitch(J) : 0; }

// census frames (usv_census.cu): interleaved like the frames, rows at a compact 16-byte pitch, padding zeroed. A census
// job's pair scratch starts with those of both cameras for every pair of a chunk (left frames, then right frames).
inline int census_pitch(const DevJob& J) { return (J.width * J.channels + 15) & ~15; }
inline size_t census_frame_bytes(const DevJob& J) { return (size_t)census_pitch(J) * J.height; }
inline size_t census_scratch_bytes_per_pair(const DevJob& J) { return J.cost_kind == USV_COST_CENSUS ? 2 * census_frame_bytes(J) : 0; }
// census frames of pairs [p0, p0 + np) of both cameras into `scratch` (one launch, counted in *n_launches), and in Jc the
// job J on them: pair 0 of Jc is pair p0 of J
cudaError_t census_chunk(const DevJob& J, int p0, int np, uint8_t* scratch, cudaStream_t st, DevJob& Jc, int* n_launches);

// x-tiles of the sliding-window sweeps (SAD and ALU correlation): 32 window positions per byte phase, the first
// 33 - tw/4 of them emitted. LeftCam windows at small x have few candidates (x' in [x - dmax, x - dmin] clipped at 0):
// the partly filled tile goes there; RightCam is the mirror image and keeps it at the high-x end.
template <class Cfg>
void set_x_tiles(const DevJob& J, Cfg& cfg) {
  cfg.stride_px = 4 * (33 - J.tw / 4);
  cfg.n_xtiles = (J.nxc + cfg.stride_px - 1) / cfg.stride_px;
  cfg.x_off = J.camera_side == USV_LEFT_CAM ? ((cfg.n_xtiles * cfg.stride_px - J.nxc) & ~3) : 0;
}

// usv_dense_corr.cu: interleaved colour frames of pairs [pair0, pair0 + np) -> planes [pair][plane][H][pitch] of both cameras
cudaError_t launch_split_planes(const DevJob& J, int pair0, int np, uint8_t* dst_l, uint8_t* dst_r, int pitch, cudaStream_t st);

// Where a dense sweep reads the rows of the chunk of np pairs from pair p0: the frames themselves (one plane), or their
// colour planes, split into `planes` (left planes first, then the right ones) by two launches counted in *n_launches.
template <class Cfg>
cudaError_t set_chunk_rows(const DevJob& J, int p0, int np, uint8_t* planes, cudaStream_t st, Cfg& cfg, int* n_launches) {
  if (J.channels == 1) {
    cfg.lp = J.left + (long long)p0 * J.frame_stride;
    cfg.rp = J.right + (long long)p0 * J.frame_stride;
    cfg.pitch = J.row_stride; cfg.plane_stride = 0; cfg.pair_stride = J.frame_stride;
    return cudaSuccess;
  }
  cfg.pitch = colour_plane_pitch(J);
  cfg.plane_stride = (long long)J.height * cfg.pitch;
  cfg.pair_stride = cfg.plane_stride * J.channels;
  uint8_t* const planes_r = planes + np * colour_planes_bytes(J);
  cfg.lp = planes; cfg.rp = planes_r;
  *n_launches += 2;
  return launch_split_planes(J, p0, np, planes, planes_r, cfg.pitch, st);
}

// sets the kernel's dynamic shared memory limit, then launches it
template <class... Params, class... Args>
cudaError_t launch_kernel(void (*k)(Params...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, const Args&... args) {
  const cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  k<<<grid, block, smem, st>>>(args...);
  return cudaGetLastError();
}

__device__ __forceinline__ unsigned long long global_timer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// candidate range (ascending x') of the window at x; mirrors include/usv_b200.h
__host__ __device__ inline void cand_range(int x, int nxc, int camera_side, int dmin, int dmax, int* lo, int* hi) {
  int a, b;
  if (camera_side == USV_LEFT_CAM) { a = x - dmax; b = x - dmin; }
  else { a = x + dmin; b = x + dmax; }
  // dmax may be "infinite" (1<<20): a stays far from int overflow for any real frame
  if (a < 0) a = 0;
  if (b > nxc - 1) b = nxc - 1;
  *lo = a; *hi = b;
}

// Disparity -> distance in cm, f64, in the reference's operation order.
//   PINHOLE : P/Main.cpp:694        ((201.6 * 4) / (disp * 0.000043)) / 1000
//   POWERLAW: P/DistanceCalculator.cpp:84
__device__ inline double distance_from_disparity(int disp, int kind) {
  if (kind == USV_DIST_PINHOLE) {
    return __ddiv_rn(__ddiv_rn(201.6 * 4, __dmul_rn((double)disp, 0.000043)), 1000.0);
  } else if (kind == USV_DIST_POWERLAW) {
    return pow(__ddiv_rn(__dmul_rn(10760.0, pow((double)disp, -0.877)), 3.0752), (1 / 0.7791));
  }
  return 0.0;
}
// The same formulas at a fractional disparity (the sub-pixel pass, usv_subpixel.cu). Kept apart from the int overload,
// whose results the integer-disparity outputs pin bit for bit.
__device__ inline double distance_from_disparity(double disp, int kind) {
  if (kind == USV_DIST_PINHOLE) {
    return __ddiv_rn(__ddiv_rn(201.6 * 4, __dmul_rn(disp, 0.000043)), 1000.0);
  } else if (kind == USV_DIST_POWERLAW) {
    return pow(__ddiv_rn(__dmul_rn(10760.0, pow(disp, -0.877)), 3.0752), (1 / 0.7791));
  }
  return 0.0;
}

// Correlation score from exact integer window sums; same formula and operation
// order as oracle/block_search_oracle.c:score_from_sums (IEEE f64, no FMA).
__device__ inline double ncc_score(long long sab, long long saa, long long sbb) {
  if (saa == 0 || sbb == 0) return 0.0;
  double ra = __drcp_rn(__dsqrt_rn((double)saa));
  double rb = __drcp_rn(__dsqrt_rn((double)sbb));
  return __dmul_rn(__dmul_rn((double)sab, ra), rb);
}
__device__ inline double zncc_score(long long n, long long sab, long long sa, long long sb, long long saa, long long sbb) {
  long long num = n * sab - sa * sb;
  long long da = n * saa - sa * sa;
  long long db = n * sbb - sb * sb;
  if (da == 0 || db == 0) return 0.0;
  double ra = __drcp_rn(__dsqrt_rn((double)da));
  double rb = __drcp_rn(__dsqrt_rn((double)db));
  return __dmul_rn(__dmul_rn((double)num, ra), rb);
}

// Normalised MatchValue of an integer cost (0 = perfect; keeps the reference's
// "accept < 0.75" meaningful, P/Main.cpp:400-401,417): the cost over its largest value.
__device__ inline double normalised_cost(uint32_t raw, int kind, int n_elems) {
  const long long unit = kind == USV_COST_SAD ? 255ll : kind == USV_COST_CENSUS ? 8ll : 65025ll;
  double den = (double)(unit * n_elems);
  return __ddiv_rn((double)raw, den);
}

// Write one window's result to every requested output array (fused epilogue:
// selection result -> Match record -> disparity -> distance).
__device__ inline void write_result(const DevJob& J, long long g, uint32_t left_index, int x, int y,
                                    int best_x, uint32_t raw, double score, double value) {
  const bool has = best_x >= 0;
  const bool accepted = has && value < J.accept_threshold;  // P/Main.cpp:417
  const int d = has ? (J.camera_side == USV_LEFT_CAM ? x - best_x : best_x - x) : 0;  // P/Main.cpp:681-693
  const uint32_t rindex = accepted ? (uint32_t)(y * J.nxc + best_x) : USV_NO_MATCH;
  double dist = 0.0;
  if (accepted && (J.out.distance || J.out.distance_f32)) {
    dist = (J.dist_lut && d >= 0 && d < J.width) ? J.dist_lut[d] : distance_from_disparity(d, J.distance_kind);
  }
  if (J.out.matches) {
    usv_match m;
    m.LeftIndex = left_index; m.RightIndex = rindex; m.MatchValue = value;
    J.out.matches[g] = m;
  }
  if (J.out.right_index) J.out.right_index[g] = rindex;
  if (J.out.raw_cost) J.out.raw_cost[g] = raw;
  if (J.out.raw_cost_u16) J.out.raw_cost_u16[g] = (uint16_t)raw;  // host checked that every cost fits; ~0 -> 0xFFFF
  if (J.out.score) J.out.score[g] = score;
  if (J.out.distance) J.out.distance[g] = dist;
  if (J.out.distance_f32) J.out.distance_f32[g] = (float)dist;
  if (J.out.disparity_u16) J.out.disparity_u16[g] = accepted ? (uint16_t)d : (uint16_t)USV_NO_DISPARITY;
}

// c + sum_{i<4} |a.byte[i] - b.byte[i]|  -> one VABSDIFF4.U8.ACC
__device__ __forceinline__ uint32_t sad4_acc(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t d;
  asm("vabsdiff4.u32.u32.u32.add %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}

// c + the Hamming distance of four census bytes -> LOP3 + POPC + IADD
__device__ __forceinline__ uint32_t hamming4_acc(uint32_t a, uint32_t b, uint32_t c) { return __popc(a ^ b) + c; }

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async8(void* smem, const void* gmem) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;\n" ::: "memory"); }

}  // namespace usv
