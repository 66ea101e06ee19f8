// usv_corr.cuh — what the three dense correlation sweeps share. They differ only in how they form Sab (usv_dense_corr.cu:
// IDP.4A sliding sums on the ALU pipes; usv_dense_mma.cu: mma.sync on the integer tensor pipe; usv_dense_umma.cu:
// tcgen05); the candidate order, the score of a candidate, the pass merge and the result of a window are stated here.
#pragma once
#include "usv_common.cuh"

namespace usv {

constexpr int kNoX = 0x7fffffff;  // x' of "no candidate yet"
// inner operation / scoring: correlation (NCC, ZNCC), SSD = Saa + Sbb - 2 Sab from the same products, or SAD with
// VABSDIFF4 in place of IDP.4A (colour frames: the gray SAD sweep has its own integer-key kernel, usv_dense.cu)
constexpr int kOpCorr = 0, kOpSsd = 1, kOpSad = 2;
constexpr int kOpSsdInt = 3;  // mma.sync kernel only: SSD scored and compared as u32 (costs below 2^28), no f64 in the inner loop

struct CorrCfg {
  const uint8_t* lp;   // planes of the left frames  [pair][plane][H][pitch]
  const uint8_t* rp;
  long long pair_stride, plane_stride;
  int pitch;           // bytes between plane rows (multiple of 4)
  const double2* stat_l;  // [pair][nyc][nxc] (-Sa, ra)
  const double2* stat_r;  // [pair][nyc][nxc] ( Sb, rb)
  double n_eff;        // n (ZNCC), 1 (NCC), 2 (SSD), -1 (SAD)
  int stride_px, n_xtiles, bh, n_bands, x_off;
  int pair0;           // first pair of this launch inside the caller's batch (outputs are indexed by the global pair)
  // tensor-pipe kernels only: running best between passes over the candidate columns, [pair][nyc][nxc]
  double* best_v;   // v = 1 - score
  double* best_sc;  // the score itself (only when the caller asked for it)
  int* best_x;
  int n_launch_pairs;  // pairs of this launch (one-dimensional grid, tile-major)
};

// (v, x') order of the reference: smaller cost v = 1 - score first, then smaller x' (P/Main.cpp:451)
__device__ __forceinline__ bool corr_v_better(double v_o, int x_o, double v_m, int x_m) { return v_o < v_m || (v_o == v_m && x_o < x_m); }
__device__ __forceinline__ bool corr_better(double sc_o, int x_o, double sc_m, int x_m) {
  return corr_v_better(__dsub_rn(1.0, sc_o), x_o, __dsub_rn(1.0, sc_m), x_m);
}

// One candidate from its Sab, n (NaN for a disparity outside [search_min, search_max]), c0 = -n * 2^52 and the
// statistics of its left window (-Sa, ra) and right position (Sb, rb), with the f64 operations of the oracle
// (oracle/block_search_oracle.c:score_from_sums) in its order:
//   n*Sab = fma(n, 2^52 + Sab, -n*2^52)   (2^52 + Sab is the u32 -> f64 conversion by bit pattern; exact)
//   num   = fma(-Sa, Sb, n*Sab)            (exact: all integers below 2^53)
//   score = (num * ra) * rb,  v = 1 - score
// Integer costs (SSD, SAD): score = (-Saa - Sbb) + n*Sab = -cost, exact, so v = 1 + cost orders by the integer cost.
struct CorrCand {
  double v, sc;
};
template <int OP>
__device__ __forceinline__ CorrCand corr_score(double n, double c0, int sab, double2 ls, double2 rs) {
  const double nsab = __fma_rn(n, __hiloint2double(0x43300000, sab), c0);
  const double num = OP != kOpCorr ? __dadd_rn(__dadd_rn(ls.x, rs.x), nsab) : __fma_rn(ls.x, rs.x, nsab);
  const double sc = OP != kOpCorr ? num : __dmul_rn(__dmul_rn(num, ls.y), rs.y);
  return {__dsub_rn(1.0, sc), sc};
}

// candidate columns [c_lo, c_hi] (ascending x', clipped to the frame) of the windows xm .. xm + n_win - 1
__device__ __forceinline__ void corr_cand_cols(const DevJob& J, bool leftcam, int xm, int n_win, int& c_lo, int& c_hi) {
  const int x_last = min(xm + n_win - 1, J.nxc - 1);
  if (leftcam) { c_lo = max(0, xm - J.dmax); c_hi = min(J.nxc - 1, x_last - J.dmin); }
  else { c_lo = max(0, xm + J.dmin); c_hi = min(J.nxc - 1, x_last + J.dmax); }
}

// Tensor-pipe kernels: merges the winner (v, sc, x') of one pass over the candidate columns with the running best of
// window e from the earlier passes. Returns true on the last pass (the winner is final); otherwise stores it.
template <bool WS>
__device__ __forceinline__ bool corr_merge_pass(const CorrCfg& cfg, long long e, int pass, int n_pass, double& v, int& xr, double& sc) {
  if (pass > 0) {
    const double vo = cfg.best_v[e];
    const int xo = cfg.best_x[e];
    if (!corr_v_better(v, xr, vo, xo)) { v = vo; xr = xo; if (WS) sc = cfg.best_sc[e]; }
  }
  if (pass < n_pass - 1) { cfg.best_v[e] = v; cfg.best_x[e] = xr; if (WS) cfg.best_sc[e] = sc; return false; }
  return true;
}

// The result of window (x, y) of pair `pair` of the caller's batch from its winner: x' (kNoX: no candidate), v and,
// for NCC / ZNCC, the score. Integer costs: raw = v - 1, exact.
template <int OP>
__device__ __forceinline__ void corr_emit(const DevJob& J, int pair, int x, int y, int xr, double v, double sc) {
  const long long w = (long long)y * J.nx + x;
  const long long g = (long long)pair * J.n_templates + w;
  if (xr == kNoX) write_result(J, g, (uint32_t)w, x, y, -1, 0xffffffffu, 0.0, __longlong_as_double(0x7ff0000000000000ll));
  else if (OP != kOpCorr) {
    const uint32_t raw = (uint32_t)__dsub_rn(v, 1.0);
    write_result(J, g, (uint32_t)w, x, y, xr, raw, 0.0, normalised_cost(raw, OP == kOpSad ? USV_COST_SAD : USV_COST_SSD, J.n_elems));
  } else write_result(J, g, (uint32_t)w, x, y, xr, 0xffffffffu, __dadd_rn(sc, 0.0), v);  // -0.0 -> 0.0 (flat windows)
}

// host side of the two tensor-pipe sweeps (usv_dense_corr.cu chooses the sweep and lays out the scratch)
using CorrKernel = void (*)(DevJob, CorrCfg);
// sets the kernel's dynamic shared memory limit, then launches it
inline cudaError_t launch_corr_kernel(CorrKernel k, dim3 grid, dim3 block, size_t smem, cudaStream_t st, const DevJob& J, const CorrCfg& cfg) {
  const cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  k<<<grid, block, smem, st>>>(J, cfg);
  return cudaGetLastError();
}
// sets cfg.bh and cfg.n_bands for cfg.n_xtiles x-tiles of np pairs on `slots` CTA slots: the band count whose grid fills
// its waves best, a band paying its th - 1 warm-up rows at `warm_weight` of a full row; bands of at most bh_cap rows
void corr_bands(const DevJob& J, CorrCfg& cfg, int np, int slots, double warm_weight, int bh_cap);
// usv_dense_mma.cu / usv_dense_umma.cu: the sweep with the products on mma.sync / tcgen05, for jobs inside the coverage
// of both (usv_dense_corr.cu: corr_tensor_supported)
cudaError_t launch_corr_mma(const DevJob& J, CorrCfg cfg, int op, int np, cudaStream_t st);
cudaError_t launch_corr_umma(const DevJob& J, CorrCfg cfg, int op, int np, cudaStream_t st);

}  // namespace usv
