// usv_dense.cu — dense stride-1 sweep for sm_100a: sliding-window SAD with a fused
// argmin + distance epilogue.
//
// Algorithm (exact in integers, identical results to the direct form):
//   h(u, d, v)  = sum_{b<4} |L[v][u+b] - R[v][u-d+b]|           one VABSDIFF4.U8.ACC
//   V(u, d, y)  = sum_{v in [y, y+th)} h(u, d, v)               kept in a register and slid
//                                                                down the rows: + new row, - old row
//   S(x, d, y)  = sum_{k < tw/4} V(x + 4k, d, y)                 SAD of window x vs candidate x-d
// so a candidate costs ~2 VABSDIFF4 + ~3 integer adds instead of tw*th/4 VABSDIFF4.
//
// Mapping. A CTA owns an x-tile (116 px for 16-px templates) x a band of output rows of one
// frame pair and walks the disparity range in passes of 8 * JT disparities. Its four warps are the four byte
// phases p = x mod 4 (packed-byte operands must be word aligned, so the shared-memory ring
// holds four byte-shifted copies of the L rows and of the R rows). Inside a warp 4 lanes run
// along x (8 window positions each) and 8 lanes along d (JT disparities each, 4 apart; the lane's
// R copy q fixes d mod 4): 8 * JT V accumulators per thread. JT = 8 (64 accumulators, 64-disparity passes,
// three CTAs per SM) serves ranges of 48 disparities and more: per thread and row the operand loads (24 words
// for 64 VABSDIFF4), the reduce-scatter, the first key, staging and barriers are paid once for twice the
// candidates; JT = 4 (32 accumulators, four CTAs per SM) serves narrow ranges. Interleaved colour frames are
// split into planes and every plane is swept into the same accumulators (NPL = 3).
// Window sums need the next x-lane's first columns: three width-4 shuffles per disparity. Keys pack
// (cost << XB | candidate code) so that "smallest cost, then smallest x'" (P/Main.cpp:451: an equal later
// candidate never replaces) is one unsigned min whatever the reduction order; the key of the next window is
// slid from the previous one with two IMADs. A reduce-scatter min over the 8 d-lanes leaves
// each lane with one window of the row, merged into the CTA's running best in shared memory.
// After the last pass the CTA decodes its keys and writes Match records / disparity / distance
// (LUT of the reference's formulas, P/Main.cpp:694 and P/DistanceCalculator.cpp:84).
//
// Why the ring is staged by threads (LDG -> funnel shift -> STS) and not by TMA: the packed-byte
// operands need byte-shifted copies, and a cp.async.bulk.tensor box must start on a 16-byte
// boundary in global memory (measured: a u8 tensor map with inner coordinate 3 raises "illegal
// instruction", coordinate 16 loads fine — scripts/dev/tma_probe.cu), as must cp.async sources.
//
// Pipes (measured on B200, profiles/microbench_r1.jsonl): VABSDIFF4/IADD3 issue at 64
// lanes/clk/SM on the ALU pipe, IMAD at 64 lanes/clk/SM on the FMA pipe in parallel,
// VIMNMX at 128. The old-row subtraction and the key slide are IMADs on purpose, to keep
// them off the ALU pipe that bounds this kernel.
#include "usv_dense_kernel.cuh"

namespace usv {

USV_DENSE_DEFINE_VARIANT(1, 4)
// usv_dense_g8.cu, usv_dense_colour.cu
template <> cudaError_t dense_launch_variant<1, 8>(int, int, bool, dim3, size_t, const DevJob&, const DenseCfg&, cudaStream_t);
template <> cudaError_t dense_launch_variant<3, 4>(int, int, bool, dim3, size_t, const DevJob&, const DenseCfg&, cudaStream_t);
template <> cudaError_t dense_launch_variant<3, 8>(int, int, bool, dim3, size_t, const DevJob&, const DenseCfg&, cudaStream_t);

static int ceil_log2(long long v) {
  int b = 0;
  while ((1ll << b) < v) ++b;
  return b;
}

// usv_dense_corr.cu: interleaved colour frames -> planes [pair][plane][H][pitch] of both cameras
cudaError_t launch_split_planes(const DevJob& J, int pair0, int np, uint8_t* dst_l, uint8_t* dst_r, int pitch, cudaStream_t st);

// scratch the colour sweep needs per pair (planes of both cameras); 0 for one-plane frames
size_t dense_scratch_bytes_per_pair(const DevJob& J) {
  return J.channels == 3 ? 2ull * 3 * J.height * colour_plane_pitch(J) : 0;
}

cudaError_t launch_dense(const DevJob& J, int n_pairs, void* d_scratch, size_t scratch_bytes, cudaStream_t st, const char** kernel_name,
                         int* n_launches) {
  // coverage of the sliding-window kernels; everything else runs on the direct-form kernel
  *n_launches = 0;
  if (J.tx || (J.channels != 1 && J.channels != 3) || J.sx != 1 || J.sy != 1) return cudaErrorNotSupported;
  if (J.cost_kind != USV_COST_SAD) return cudaErrorNotSupported;
  const int nw = J.tw / 4;
  if (J.tw % 4 != 0 || !(nw == 2 || nw == 3 || nw == 4 || nw == 6 || nw == 8) || J.th > 64) return cudaErrorNotSupported;
  const int npl = J.channels;
  DenseCfg cfg;
  cfg.stride_px = 4 * (32 - nw + 1);
  cfg.n_xtiles = (J.nxc + cfg.stride_px - 1) / cfg.stride_px;
  // LeftCam windows at small x have few candidates (x' in [x - dmax, x - dmin] clipped at 0): put the
  // partly filled tile there; RightCam is the mirror image and keeps it at the high-x end
  cfg.x_off = J.camera_side == USV_LEFT_CAM ? ((cfg.n_xtiles * cfg.stride_px - J.nxc) & ~3) : 0;
  cfg.xb = ceil_log2((long long)J.nxc + kCodeOff + 1);
  const long long smax = 255ll * J.n_elems;
  if (ceil_log2(smax + 1) + cfg.xb > 31) return cudaErrorNotSupported;  // bit 31 marks invalid candidates
  // bands: as tall as shared memory allows (amortises the th-1 warm-up rows), but enough CTAs to fill 148 SMs
  const bool wide_range = std::min(J.dmax, J.nxc - 1) - std::max(J.dmin, -(J.nxc - 1)) + 1 >= 48;
  // 8 disparities per thread (64 per pass, 64 accumulators, three CTAs per SM) when the range is wide enough to fill such
  // passes, gray and colour alike: 24 operand words for 64 VABSDIFF4 instead of 20 for 32, half the reduce-scatter, staging and
  // barriers per candidate (measured on C2: 10.08 against 10.92 ms although the full-range triangle wastes more slots)
  const int jt = wide_range ? 8 : 4;
  const int smem_budget = (npl == 1 && jt == 4) ? 56 * 1024 : 75 * 1024;  // 4 CTAs / SM; colour: 3 (one more plane set of temporaries in registers)
  const bool ring2 = npl > 1 || J.th > 16;  // measured: the short double-fetched ring pays from 24-row templates on
  const int rb = npl == 1 ? 4 : 2;
  cfg.ring_words = (ring2 ? 4 * rb : J.th + 2 * rb) * npl * row_words(jt);
  int bh_max = (smem_budget - cfg.ring_words * 4) / 512;
  if (bh_max < 8) return cudaErrorNotSupported;
  const int ctas_per_sm = (npl == 1 && jt == 4) ? 4 : 3;
  int n_bands = (J.nyc + bh_max - 1) / bh_max;
  while ((long long)n_bands * cfg.n_xtiles * n_pairs < g_sm_count * (ctas_per_sm - 1) && n_bands < (J.nyc + 15) / 16) ++n_bands;
  cfg.bh = (J.nyc + n_bands - 1) / n_bands;
  cfg.n_bands = (J.nyc + cfg.bh - 1) / cfg.bh;
  const size_t smem = (size_t)cfg.ring_words * 4 + (size_t)cfg.bh * 512;
  const int pitch = npl == 1 ? J.row_stride : colour_plane_pitch(J);
  cfg.pitch = pitch;
  cfg.plane_stride = npl == 1 ? 0 : (long long)J.height * pitch;
  cfg.pair_stride = npl == 1 ? J.frame_stride : cfg.plane_stride * npl;
  cfg.chunk_pairs = (int)std::min<long long>(64, std::max<long long>(1, (48ll << 20) / (2ll * npl * J.height * pitch)));
  // colour: the planes of a chunk of pairs live in the caller's scratch
  const size_t per_pair = dense_scratch_bytes_per_pair(J);
  if (npl > 1 && (!d_scratch || scratch_bytes < per_pair)) return cudaErrorNotSupported;
  const int launch_pairs = npl == 1 ? n_pairs : (int)std::min<size_t>((size_t)n_pairs, scratch_bytes / per_pair);
  if ((long long)cfg.n_xtiles * cfg.n_bands * launch_pairs > 0x7fffffffll) return cudaErrorNotSupported;
  for (int p0 = 0; p0 < n_pairs; p0 += launch_pairs) {
    const int np = std::min(launch_pairs, n_pairs - p0);
    cfg.n_pairs = np;
    cfg.pair0 = p0;
    if (npl == 1) {
      cfg.lp = J.left; cfg.rp = J.right;
    } else {
      uint8_t* pl_l = (uint8_t*)d_scratch;
      uint8_t* pl_r = pl_l + (size_t)np * cfg.pair_stride;
      cudaError_t e = launch_split_planes(J, p0, np, pl_l, pl_r, pitch, st);
      if (e != cudaSuccess) return e;
      cfg.lp = pl_l; cfg.rp = pl_r;
      *n_launches += 2;
    }
    const dim3 grid(cfg.n_xtiles * cfg.n_bands * np);
    const int dir = J.camera_side == USV_LEFT_CAM ? -1 : 1;
    const cudaError_t e = npl == 3 ? (jt == 8 ? dense_launch_variant<3, 8>(dir, nw, ring2, grid, smem, J, cfg, st)
                                              : dense_launch_variant<3, 4>(dir, nw, ring2, grid, smem, J, cfg, st))
                          : jt == 8 ? dense_launch_variant<1, 8>(dir, nw, ring2, grid, smem, J, cfg, st)
                                    : dense_launch_variant<1, 4>(dir, nw, ring2, grid, smem, J, cfg, st);
    if (e != cudaSuccess) return e;
    *n_launches += 1;
  }
  *kernel_name = "dense_sad_argmin_kernel";
  return cudaSuccess;
}


}  // namespace usv
