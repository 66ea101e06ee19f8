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
//
// USV_COST_CENSUS runs the same sweep over census frames (usv_census.cu), transformed into the pair scratch once per chunk
// of pairs, as dense_census_argmin_kernel: h(u, d, v) = popc(L ^ R) of one packed word (LOP3 + POPC + IADD instead of
// one VABSDIFF4), at most 8 per byte where SAD has 255.
#include "usv_dense_kernel.cuh"

namespace usv {

// compiled in usv_dense_g8.cu, usv_dense_colour.cu, usv_dense_census.cu and usv_dense_census_colour.cu
extern template DenseKernel dense_kernel<1, 8>(int, int, bool);
extern template DenseKernel dense_kernel<3, 4>(int, int, bool);
extern template DenseKernel dense_kernel<3, 8>(int, int, bool);
extern template DenseKernel dense_kernel<1, 4, true>(int, int, bool);
extern template DenseKernel dense_kernel<1, 8, true>(int, int, bool);
extern template DenseKernel dense_kernel<3, 4, true>(int, int, bool);
extern template DenseKernel dense_kernel<3, 8, true>(int, int, bool);

static int ceil_log2(long long v) {
  int b = 0;
  while ((1ll << b) < v) ++b;
  return b;
}

// Shared memory of a CTA: the row ring, then bands of up to bh_max rows of 128 keys. 4 CTAs per SM for gray JT = 4,
// otherwise 3 (colour: one more plane set of temporaries in registers).
constexpr int dense_smem_budget(int npl, int jt) { return npl == 1 && jt == 4 ? 56 * 1024 : 75 * 1024; }
constexpr int dense_ring_words(int npl, int jt, bool ring2, int th) {
  return (ring2 ? 4 * (npl == 1 ? 4 : 2) : th + 2 * 4) * npl * row_words(jt);
}
constexpr int dense_bh_max(int npl, int jt, bool ring2, int th) { return (dense_smem_budget(npl, jt) - 4 * dense_ring_words(npl, jt, ring2, th)) / 512; }
// the tallest rings: th + 8 rows of one plane (th <= 16; the two-half ring holds 16) and 8 rows of three planes
static_assert(dense_bh_max(1, 4, false, 16) >= 8 && dense_bh_max(1, 8, false, 16) >= 8 && dense_bh_max(3, 4, true, 0) >= 8 &&
                  dense_bh_max(3, 8, true, 0) >= 8,
              "bands of at least 8 rows");

// The SAD sweep's launch of a dense stride-1 SAD or census job of one or three planes (usv_capi.cu: plan_match checks
// those), for a batch of n_pairs; false when the sweep does not cover the job.
struct DenseLaunch {
  DenseCfg cfg;  // all but the pairs of a launch and where its rows come from
  int jt;
  bool ring2;
  size_t smem;
};
static bool dense_launch_cfg(const DevJob& J, int n_pairs, DenseLaunch& L) {
  const int nw = J.tw / 4, npl = J.channels;
  const bool census = J.cost_kind == USV_COST_CENSUS;
  if ((J.cost_kind != USV_COST_SAD && !census) || J.tw % 4 != 0 || !(nw == 2 || nw == 3 || nw == 4 || nw == 6 || nw == 8) || J.th > 64) return false;
  DenseCfg& cfg = L.cfg;
  set_x_tiles(J, cfg);
  cfg.xb = ceil_log2((long long)J.nxc + kCodeOff + 1);
  // bit 31 marks invalid candidates. Census (at most 8 a byte): at th <= 64 any frame narrower than 2^15 px fits
  if (ceil_log2((census ? 8ll : 255ll) * J.n_elems + 1) + cfg.xb > 31) return false;
  // bands: as tall as shared memory allows (amortises the th-1 warm-up rows), but enough CTAs to fill 148 SMs
  const bool wide_range = std::min(J.dmax, J.nxc - 1) - std::max(J.dmin, -(J.nxc - 1)) + 1 >= 48;
  // 8 disparities per thread (64 per pass, 64 accumulators, three CTAs per SM) when the range is wide enough to fill such
  // passes, gray and colour alike: 24 operand words for 64 VABSDIFF4 instead of 20 for 32, half the reduce-scatter, staging and
  // barriers per candidate (measured on C2: 10.08 against 10.92 ms although the full-range triangle wastes more slots)
  L.jt = wide_range ? 8 : 4;
  L.ring2 = npl > 1 || J.th > 16;  // measured: the short double-fetched ring pays from 24-row templates on
  cfg.ring_words = dense_ring_words(npl, L.jt, L.ring2, J.th);
  const int bh_max = dense_bh_max(npl, L.jt, L.ring2, J.th);
  const int ctas_per_sm = (npl == 1 && L.jt == 4) ? 4 : 3;
  int n_bands = (J.nyc + bh_max - 1) / bh_max;
  while ((long long)n_bands * cfg.n_xtiles * n_pairs < g_sm_count * (ctas_per_sm - 1) && n_bands < (J.nyc + 15) / 16) ++n_bands;
  cfg.bh = (J.nyc + n_bands - 1) / n_bands;
  cfg.n_bands = (J.nyc + cfg.bh - 1) / cfg.bh;
  L.smem = (size_t)cfg.ring_words * 4 + (size_t)cfg.bh * 512;
  const int pitch = npl == 1 ? J.row_stride : colour_plane_pitch(J);
  cfg.chunk_pairs = (int)std::min<long long>(64, std::max<long long>(1, (48ll << 20) / (2ll * npl * J.height * pitch)));
  // one-dimensional grid of the whole batch. Tiles of at least 100 px and bands of at least 16 rows give a pair at most
  // about nxc * nyc / 1600 blocks, so 2^31 of them would need some 3.4e12 pixels of resident frames per camera
  return (long long)cfg.n_xtiles * cfg.n_bands * n_pairs <= 0x7fffffffll;
}

bool dense_sad_covers(const DevJob& J, int n_pairs) {
  DenseLaunch L;
  return dense_launch_cfg(J, n_pairs, L);
}

// scratch the sweep needs per pair: the census frames (census) and the colour planes of both cameras
size_t dense_scratch_bytes_per_pair(const DevJob& J) { return census_scratch_bytes_per_pair(J) + 2 * colour_planes_bytes(J); }

// census frames and colour planes of a chunk of pairs live in the caller's scratch, which holds at least one pair's
cudaError_t launch_dense(const DevJob& J, int n_pairs, void* d_scratch, size_t scratch_bytes, cudaStream_t st, int* n_launches) {
  DenseLaunch L;
  if (!dense_launch_cfg(J, n_pairs, L)) return cudaErrorInvalidValue;
  const int dir = J.camera_side == USV_LEFT_CAM ? -1 : 1, nw = J.tw / 4;
  const bool census = J.cost_kind == USV_COST_CENSUS;
  const DenseKernel k =
      census ? (J.channels == 3 ? (L.jt == 8 ? dense_kernel<3, 8, true>(dir, nw, L.ring2) : dense_kernel<3, 4, true>(dir, nw, L.ring2))
                                : (L.jt == 8 ? dense_kernel<1, 8, true>(dir, nw, L.ring2) : dense_kernel<1, 4, true>(dir, nw, L.ring2)))
             : (J.channels == 3 ? (L.jt == 8 ? dense_kernel<3, 8>(dir, nw, L.ring2) : dense_kernel<3, 4>(dir, nw, L.ring2))
                                : (L.jt == 8 ? dense_kernel<1, 8>(dir, nw, L.ring2) : dense_kernel<1, 4>(dir, nw, L.ring2)));
  const size_t per_pair = dense_scratch_bytes_per_pair(J);
  const int chunk = per_pair ? (int)std::min<size_t>((size_t)n_pairs, scratch_bytes / per_pair) : n_pairs;
  DenseCfg cfg = L.cfg;
  for (int p0 = 0; p0 < n_pairs; p0 += chunk) {
    const int np = std::min(chunk, n_pairs - p0);
    cfg.n_pairs = np;
    cfg.pair0 = p0;
    // census: the chunk's census frames first (the sweep then reads them from pair 0 of Jc), its colour planes after them
    DevJob Jc = J;
    uint8_t* planes = (uint8_t*)d_scratch;
    cudaError_t e = cudaSuccess;
    if (census) {
      e = census_chunk(J, p0, np, planes, st, Jc, n_launches);
      planes += np * census_scratch_bytes_per_pair(J);
    }
    if (e == cudaSuccess) e = set_chunk_rows(Jc, census ? 0 : p0, np, planes, st, cfg, n_launches);
    if (e == cudaSuccess) e = launch_kernel(k, dim3(cfg.n_xtiles * cfg.n_bands * np), dim3(kDenseThreads), L.smem, st, Jc, cfg, 0xffffffffu);
    if (e != cudaSuccess) return e;
    *n_launches += 1;
  }
  return cudaSuccess;
}

}  // namespace usv
