// usv_dense_mma.cu — dense stride-1 sweep for NCC / ZNCC / SSD with the row products on the integer tensor pipe
// (IMMA.16832.U8.U8 / IMMA.16816.U8.U8 through mma.sync; measured on this pool's B200: 1 950 MAC/clk/SM, 7.6x the
// IDP.4A rate of the ALU path in usv_dense_corr.cu — scripts/dev/imma_probe.cu, profiles/imma_probe_r1.jsonl).
//
// The correlation recast as a contraction (BASELINE north_star (1): "tensor cores only if the NCC correlation is
// recast as a dense contraction and ncu shows it beats the ALU path"). For one image row v of one colour plane
//     G_v[x, x'] = sum_{c < tw} L[v][x + c] * R[v][x' + c]
// is a product of two Toeplitz matrices, A[x][c] = L[v][x + c] (16 windows x tw bytes) and B[c][x'] = R[v][x' + c]
// (tw bytes x 8 candidates): one mma.m16n8k32 (tw <= 32) or m16n8k16 (tw <= 16) per (16 windows, 8 candidates, plane);
// the bytes of A beyond a narrower template are zeroed.
// A fragment register of either operand is four consecutive bytes of the row at an arbitrary byte offset, i.e. one
// word of one of the four byte-shifted copies of the row that the ALU kernels already keep in shared memory — no
// im2col is ever materialised. Sab(x, x', y) = sum over the th rows of the window and the planes of G_v is slid down
// the rows in the s32 accumulators exactly like the ALU kernels slide V: + the entering row, - the leaving row
// (products are u8 x u8, so the leaving row goes through a zeroed temporary and an integer subtract). All sums are
// exact integers, and the score is computed from them by the same f64 operations in the same order as
// oracle/block_search_oracle.c:score_from_sums (see usv_dense_corr.cu), so scores, costs and indices stay bit-exact.
//
// Mapping. CTA = 32 windows (x-tile) x a band of output rows x one pair, 8 warps = 2 m16 tiles x 4 quarters of the
// pass's 288 candidate columns: a warp owns 16 windows x 72 columns = 9 n8-tiles (36 accumulators per thread). The
// candidates of the 32 windows are the parallelogram x' in [x - dmax, x - dmin] (LeftCam) inside a rectangle of
// 32 + D - 1 columns: D = 256 needs one pass of 287 columns, 89 % of the products are wanted. Groups of three tiles
// that lie wholly outside the parallelogram are skipped (warp-uniform), entries outside it are masked by an unsigned
// range test on d, entries outside the frame carry NaN statistics.
// Per row: barrier; global loads of the next row's ring words into registers, cp.async of its window statistics; one
// warp merges the four quarters' winners of the previous row and writes the results (fused epilogue: Match /
// disparity / distance); products of the entering and of the leaving row; f64 scores and running best over the
// thread's 36 candidates of 2 windows; 2 shuffles across the quad; the staged registers go to shared memory.
// Several passes (wide ranges) keep the running best per window in a global scratch array between passes.
#include <algorithm>
#include <cstdlib>
#include <type_traits>

#include "usv_corr.cuh"

namespace usv {

constexpr int kMThreads = 256;
constexpr int kMWin = 32;                 // windows per CTA: two m16 tiles
constexpr int kNTW = 9;                   // n8 tiles per warp and pass
constexpr int kNG = 3;                    // tiles per group (the unit of skipping and of the scoring blocks)
constexpr int kWarpCols = 8 * kNTW;       // 72
constexpr int kPassCols = 4 * kWarpCols;  // 288 candidate columns per pass
constexpr int kMLW = 24;                  // words per L copy (17 used; 24 keeps the four copies on disjoint banks)
constexpr int kMRW = 88;                  // words per R copy (81 used; 88 = 24 mod 32 likewise)
constexpr int kMLChunks = 5, kMRChunks = 21;  // 16-byte chunks staged per row: L 20 words, R 84 words
constexpr int kMRowWords = 4 * kMLW + 4 * kMRW;  // one (slot, plane): 4 L copies + 4 R copies

__device__ __forceinline__ void imma_k32(int (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k32.row.col.s32.u8.u8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void imma_k16(int (&c)[4], uint32_t a0, uint32_t a1, uint32_t b0) {
  asm("mma.sync.aligned.m16n8k16.row.col.s32.u8.u8.s32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%0,%1,%2,%3};"
      : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3])
      : "r"(a0), "r"(a1), "r"(b0));
}

// TW = K of one product (16 or 32; the template is tw <= TW bytes wide); WS: the caller asked for the f64 score of the winner (otherwise
// only v = 1 - score, the MatchValue, is tracked). The camera side is a run-time sign: LeftCam x' = x - d, RightCam x + d.
template <int TW, int NPL, int OP, bool WS>
__global__ void __launch_bounds__(kMThreads, 2) dense_corr_mma_kernel(const DevJob J, const CorrCfg cfg) {
  constexpr bool ISSD = OP == kOpSsdInt;  // integer scoring: cost = Saa + Sbb - 2 Sab in u32
  constexpr int NB = TW == 32 ? kNTW + 2 : kNTW;  // B words a thread reads per plane row (k32: b1 of tile j = b0 of tile j + 2)
  constexpr int NA = TW == 32 ? 4 : 2;            // A words
  extern __shared__ __align__(16) uint32_t smem_u32[];
  uint32_t* s_ring = smem_u32;                                                   // [enter, leave][2 slots][NPL][kMRowWords]
  double2* s_rs = reinterpret_cast<double2*>(s_ring + 4 * NPL * kMRowWords);     // [2][kPassCols] (Sb, rb) of the output row
  double2* s_ls = s_rs + 2 * kPassCols;                                          // [2][32] (-Sa, ra) of the CTA's windows
  double* s_mv = reinterpret_cast<double*>(s_ls + 2 * kMWin);                    // [2][4 quarters][32 windows] best v
  double* s_msc = s_mv + 2 * 4 * kMWin;                                          // [2][4][32] its score (WS)
  int* s_mx = reinterpret_cast<int*>(s_msc + 2 * 4 * kMWin);                     // [2][4][32] its x'

  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, g = lane >> 2, t = lane & 3;
  const int q = w & 3, mi = w >> 2;  // quarter of the pass's columns, m16 tile
  // one-dimensional grid, the longest CTAs first: an x-tile's work grows with the candidate columns its windows can reach
  // (LeftCam: with x), so all CTAs of the heaviest tile are dispatched first and the lightest fill the tail (with bounded
  // ranges this tail is worth more than the L2 locality of chunks of pairs: C3 2.65k pairs/s against 2.53k with 8-pair chunks)
  const int per_tile = cfg.n_bands * cfg.n_launch_pairs;
  const int t_ord = blockIdx.x / per_tile, t_rem = blockIdx.x - t_ord * per_tile;
  const int tile = J.camera_side == USV_LEFT_CAM ? cfg.n_xtiles - 1 - t_ord : t_ord;
  const int pair = t_rem / cfg.n_bands, band = t_rem - pair * cfg.n_bands;
  const int xm = kMWin * tile;
  const int y0 = band * cfg.bh;
  const int bh = min(cfg.bh, J.nyc - y0);
  const int th = J.th;
  const int rows_in = bh + th - 1;
  const int nxc = J.nxc;
  const int row_words = cfg.pitch >> 2;
  const bool leftcam = J.camera_side == USV_LEFT_CAM;
  const uint8_t* Lb = cfg.lp + (long long)pair * cfg.pair_stride + (long long)y0 * cfg.pitch;
  const uint8_t* Rb = cfg.rp + (long long)pair * cfg.pair_stride + (long long)y0 * cfg.pitch;
  const double2* stl = cfg.stat_l + (long long)pair * J.nyc * nxc;
  const double2* str = cfg.stat_r + (long long)pair * J.nyc * nxc;
  const double nan = __longlong_as_double(0x7ff8000000000000ll);
  const double inf = __longlong_as_double(0x7ff0000000000000ll);
  const uint32_t dspan = (uint32_t)(J.dmax - J.dmin);

  int c_lo, c_hi;
  corr_cand_cols(J, leftcam, xm, kMWin, c_lo, c_hi);
  const int col_base = c_lo & ~7;
  const int n_pass = c_hi >= c_lo ? (c_hi - col_base) / kPassCols + 1 : 1;

  // ---- staging: a task = one 16-byte chunk of one plane row of one half (entering / leaving): five aligned global
  // words -> the four byte-shifted copies; task tid. The window statistics of the next output row go from global to
  // shared memory by cp.async (no registers): 288 right positions + 32 left windows.
  constexpr int kChunks = kMLChunks + kMRChunks;
  constexpr int kTasks = 2 * NPL * kChunks;
  static_assert(kTasks <= kMThreads - 96 && kPassCols == 3 * 96, "ring tasks on warps 0..4, statistics on warps 5..7");
  const bool t_on = tid < kTasks;
  const int t_half = tid / (NPL * kChunks), t_hrem = tid - t_half * (NPL * kChunks);
  const int t_pl = t_hrem / kChunks, t_c = t_hrem - t_pl * kChunks;
  const bool t_left = t_c < kMLChunks;
  const int t_w0 = 4 * (t_left ? t_c : t_c - kMLChunks);
  const uint32_t* t_gp = reinterpret_cast<const uint32_t*>((t_left ? Lb : Rb) + (long long)t_pl * cfg.plane_stride);
  const int t_kw = t_left ? kMLW : kMRW, t_back = t_half ? th : 0;
  const int t_off = (t_half * 2 * NPL + t_pl) * kMRowWords + (t_left ? 0 : 4 * kMLW) + t_w0;
  uint32_t pw[5];   // prefetched ring words
  int t_idx[5];     // word offsets inside the plane row, clamped to the row (set per pass: the R chunks move with it)
  const uint32_t* t_row = nullptr;  // the plane row the next prefetch reads (advances one row per call)
  auto prefetch = [&](int r, int xcol0) {
    if (t_on && r >= t_back) {
#pragma unroll
      for (int k = 0; k < 5; ++k) pw[k] = __ldg(t_row + t_idx[k]);
      t_row += row_words;
    }
    if (r >= th - 1 && tid >= kMThreads - 96) {  // warps 5..7: warps 0..4 carry the ring tasks
      const long long ro = (long long)(y0 + r - (th - 1)) * nxc;
      const int slot = r & 1, i = tid - (kMThreads - 96);
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const int col = i + k * 96, xk = xcol0 + col;
        // a candidate outside the frame loses every comparison: NaN statistics
        if (xk > nxc - 1) s_rs[slot * kPassCols + col] = make_double2(nan, nan);
        else cp_async16(&s_rs[slot * kPassCols + col], str + ro + xk);
      }
      if (i < kMWin) cp_async16(&s_ls[slot * kMWin + i], stl + ro + min(xm + i, nxc - 1));
    }
    cp_async_commit();
  };
  auto store_staged = [&](int r) {
    if (t_on && r - t_back >= 0) {
      uint32_t* dst = s_ring + (r & 1) * NPL * kMRowWords + t_off;
      *reinterpret_cast<uint4*>(dst) = make_uint4(pw[0], pw[1], pw[2], pw[3]);
#pragma unroll
      for (int s = 1; s < 4; ++s)
        *reinterpret_cast<uint4*>(dst + s * t_kw) = make_uint4(__funnelshift_r(pw[0], pw[1], 8 * s), __funnelshift_r(pw[1], pw[2], 8 * s),
                                                               __funnelshift_r(pw[2], pw[3], 8 * s), __funnelshift_r(pw[3], pw[4], 8 * s));
    }
    cp_async_wait_all();
  };

  // fragment words of this thread inside a (slot, plane): operand byte = base + g + 4t (+8 for row g + 8, +16 for the
  // upper half of K): copy g & 3, word (g >> 2) + t + ...
  const int a_off = (g & 3) * kMLW + 4 * mi + (g >> 2) + t;
  // templates narrower than K: the bytes of A beyond the template width are zeroed (k = 4t + i, + 16 for the upper words)
  auto byte_mask = [](int n) { return n >= 4 ? 0xffffffffu : n <= 0 ? 0u : (1u << (8 * n)) - 1u; };
  const uint32_t a_mask_lo = byte_mask(J.tw - 4 * t), a_mask_hi = byte_mask(J.tw - 16 - 4 * t);
  const int b_off = 4 * kMLW + (g & 3) * kMRW + 2 * kNTW * q + (g >> 2) + t;

  // one warp per row merges the four quarters' winners and writes the results (last pass) or the running best
  auto merge_row = [&](int r, int pass) {
    if (w != 5 + r % 3) return;
    const int par = r & 1;
    const int x = xm + lane, yo = y0 + r - (th - 1);
    double v = s_mv[(par * 4 + 0) * kMWin + lane], sc = WS ? s_msc[(par * 4 + 0) * kMWin + lane] : 0.0;
    int xr = s_mx[(par * 4 + 0) * kMWin + lane];
#pragma unroll
    for (int qq = 1; qq < 4; ++qq) {
      const double vo = s_mv[(par * 4 + qq) * kMWin + lane];
      const int xo = s_mx[(par * 4 + qq) * kMWin + lane];
      if (corr_v_better(vo, xo, v, xr)) { v = vo; xr = xo; if (WS) sc = s_msc[(par * 4 + qq) * kMWin + lane]; }
    }
    if (x > nxc - 1) return;
    if (corr_merge_pass<WS>(cfg, ((long long)pair * J.nyc + yo) * nxc + x, pass, n_pass, v, xr, sc))
      corr_emit<OP>(J, cfg.pair0 + pair, x, yo, xr, v, sc);
  };

  for (int pass = 0; pass < n_pass; ++pass) {
    const int xcol0 = col_base + pass * kPassCols;
    const int wcol0 = xcol0 + kWarpCols * q;  // first column of this warp
    const int xc0 = wcol0 + 2 * t;            // x' of this thread's entry (tile 0, el 0)
    // groups of kNG tiles (16 windows x 24 columns) against the parallelogram dmin <= d <= dmax and the columns
    // [c_lo, c_hi]: bit jg of any_g = some entry may be a candidate. Skipping is only an optimisation: the range test
    // on d and the NaN statistics of out-of-frame columns reject every entry of a skipped group.
    const int xa = xm + 16 * mi;
    uint32_t any_g = 0u, full_g = 0u;  // full: every entry of the group has d in range, the test is skipped
#pragma unroll
    for (int jg = 0; jg < kNTW / kNG; ++jg) {
      const int cb = wcol0 + 8 * kNG * jg, ce = cb + 8 * kNG - 1;
      const int d_lo = leftcam ? xa - ce : cb - xa - 15, d_hi = leftcam ? xa + 15 - cb : ce - xa;
      if (c_hi >= c_lo && cb <= c_hi && ce >= c_lo && d_hi >= J.dmin && d_lo <= J.dmax && xa <= nxc - 1) {
        any_g |= 1u << jg;
        if (d_lo >= J.dmin && d_hi <= J.dmax) full_g |= 1u << jg;
      }
    }
    // d - dmin of the thread's entry (eh, tile 0, el 0); tile j, el move it by -/+ (8 j + el)
    int ub[2];
#pragma unroll
    for (int eh = 0; eh < 2; ++eh) {
      const int x = xa + g + 8 * eh;
      ub[eh] = (leftcam ? x - xc0 : xc0 - x) - J.dmin;
    }
    const int usgn = leftcam ? -1 : 1;
    int acc[kNTW][4];
#pragma unroll
    for (int j = 0; j < kNTW; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[j][e] = 0;

    {
      const int gb = ((t_left ? xm : xcol0) >> 2) + t_w0;
#pragma unroll
      for (int k = 0; k < 5; ++k) t_idx[k] = min(max(gb + k, 0), row_words - 1);
      t_row = t_gp;  // the first call that loads is r = t_back: row r - t_back = 0 of the band
    }
    __syncthreads();  // the previous pass is done with the ring and the merge buffers
    prefetch(0, xcol0);
    store_staged(0);
    for (int r = 0; r < rows_in; ++r) {
      __syncthreads();  // row r staged; every warp finished row r - 1
      const bool more = r + 1 < rows_in;
      if (more) prefetch(r + 1, xcol0);
      if (r >= th) merge_row(r - 1, pass);
      const uint32_t* ring_e = s_ring + (r & 1) * NPL * kMRowWords;
      // G of one ring row (all planes) added into c: plane by plane, the B words slide along the tiles
      auto row_products = [&](const uint32_t* ring, int (&c)[kNTW][4]) {
#pragma unroll
        for (int pl = 0; pl < NPL; ++pl) {
          const uint32_t* ap = ring + pl * kMRowWords + a_off;
          const uint32_t* bp = ring + pl * kMRowWords + b_off;
          uint32_t a[4], b[NB];
#pragma unroll
          for (int k = 0; k < NA; ++k) a[k] = ap[2 * k] & (k < 2 ? a_mask_lo : a_mask_hi);
#pragma unroll
          for (int j = 0; j < NB; ++j) b[j] = bp[2 * j];
#pragma unroll
          for (int jg = 0; jg < kNTW / kNG; ++jg)
            if (any_g >> jg & 1) {
#pragma unroll
              for (int jj = 0; jj < kNG; ++jj) {
                const int j = kNG * jg + jj;
                if (TW == 32) imma_k32(c[j], a[0], a[1], a[2], a[3], b[j], b[TW == 32 ? j + 2 : j]);
                else imma_k16(c[j], a[0], a[1], b[j]);
              }
            }
        }
      };
      // ---- entering row: acc += G_r
      row_products(ring_e, acc);
      // ---- leaving row: acc -= G_{r - th} (u8 x u8 products: through a zeroed temporary)
      if (r >= th) {
        int tmp[kNTW][4];
#pragma unroll
        for (int j = 0; j < kNTW; ++j)
#pragma unroll
          for (int e = 0; e < 4; ++e) tmp[j][e] = 0;
        row_products(ring_e + 2 * NPL * kMRowWords, tmp);
#pragma unroll
        for (int j = 0; j < kNTW; ++j)
#pragma unroll
          for (int e = 0; e < 4; ++e) acc[j][e] -= tmp[j][e];
      }
      // ---- scores of the output row and the running best of the thread's two windows over its 36 candidates
      if (r >= th - 1) {
        const int par = r & 1;
        const double n_eff = cfg.n_eff, c0 = __dmul_rn(cfg.n_eff, -4503599627370496.0);
        double2 La[2];
        double bv[2], bs[2];
        int bi[2];
#pragma unroll
        for (int eh = 0; eh < 2; ++eh) {
          La[eh] = s_ls[par * kMWin + 16 * mi + 8 * eh + g];
          bv[eh] = inf;
          bs[eh] = -inf;
          bi[eh] = -1;
        }
        const double2* rs = s_rs + par * kPassCols + kWarpCols * q + 2 * t;
        if (ISSD) {
          // SSD as integers: the statistics hold (-Saa, 1) / (-Sbb, 1) (NaN outside the frame), so
          // cost = Saa + Sbb - 2 Sab < 2^28 (checked on the host); a column outside the frame contributes 2^30 and
          // its cost stays above 2^29, i.e. above every real one, and is discarded after the loop
          uint32_t kw[2], bc[2] = {0xffffffffu, 0xffffffffu};
#pragma unroll
          for (int eh = 0; eh < 2; ++eh) kw[eh] = __double2uint_rn(-La[eh].x);
#pragma unroll
          for (int jg = 0; jg < kNTW / kNG; ++jg)
            if (any_g >> jg & 1) {
              uint32_t cc[kNG][2][2];
#pragma unroll
              for (int jj = 0; jj < kNG; ++jj) {
                const int j = kNG * jg + jj;
                const double r0 = rs[8 * j].x, r1 = rs[8 * j + 1].x;
                const uint32_t sb0 = r0 != r0 ? (1u << 30) : __double2uint_rn(-r0), sb1 = r1 != r1 ? (1u << 30) : __double2uint_rn(-r1);
#pragma unroll
                for (int eh = 0; eh < 2; ++eh)
#pragma unroll
                  for (int el = 0; el < 2; ++el)
                    cc[jj][eh][el] = kw[eh] + (el ? sb1 : sb0) - 2u * (uint32_t)acc[j][2 * eh + el];
              }
              auto update = [&](auto masked_t) {
#pragma unroll
                for (int jj = 0; jj < kNG; ++jj)
#pragma unroll
                  for (int eh = 0; eh < 2; ++eh)
#pragma unroll
                    for (int el = 0; el < 2; ++el) {  // ascending x': a later equal candidate never replaces
                      const int idx = 8 * (kNG * jg + jj) + el;
                      bool take = cc[jj][eh][el] < bc[eh];
                      if (decltype(masked_t)::value) take = take && (uint32_t)(ub[eh] + usgn * idx) <= dspan;
                      if (take) { bc[eh] = cc[jj][eh][el]; bi[eh] = idx; }
                    }
              };
              if (full_g >> jg & 1) update(std::false_type{});
              else update(std::true_type{});
            }
#pragma unroll
          for (int eh = 0; eh < 2; ++eh) {
            const bool none = bc[eh] >= (1u << 29);
            bv[eh] = none ? inf : __dadd_rn(1.0, (double)bc[eh]);  // v = 1 + SSD, as the f64 path carries it
            if (none) bi[eh] = -1;
          }
        } else {
#pragma unroll
        for (int jg = 0; jg < kNTW / kNG; ++jg)
          if (any_g >> jg & 1) {
            double vv[kNG][2][2], ss[kNG][2][2];
#pragma unroll
            for (int jj = 0; jj < kNG; ++jj) {
              const int j = kNG * jg + jj;
              const double2 R0 = rs[8 * j], R1 = rs[8 * j + 1];
#pragma unroll
              for (int eh = 0; eh < 2; ++eh)
#pragma unroll
                for (int el = 0; el < 2; ++el) {
                  const double2 Rr = el ? R1 : R0;
                  const CorrCand c = corr_score<OP>(n_eff, c0, acc[j][2 * eh + el], La[eh], Rr);
                  ss[jj][eh][el] = c.sc;
                  vv[jj][eh][el] = c.v;
                }
            }
            // ascending x': a later equal candidate never replaces (P/Main.cpp:451)
            auto update = [&](auto masked_t) {
#pragma unroll
              for (int jj = 0; jj < kNG; ++jj)
#pragma unroll
                for (int eh = 0; eh < 2; ++eh)
#pragma unroll
                  for (int el = 0; el < 2; ++el) {
                    const int idx = 8 * (kNG * jg + jj) + el;
                    bool take = vv[jj][eh][el] < bv[eh];
                    if (decltype(masked_t)::value) take = take && (uint32_t)(ub[eh] + usgn * idx) <= dspan;
                    if (take) { bv[eh] = vv[jj][eh][el]; bi[eh] = idx; if (WS) bs[eh] = ss[jj][eh][el]; }
                  }
            };
            if (full_g >> jg & 1) update(std::false_type{});
            else update(std::true_type{});
          }
        }
        // best over the quad (the four t-lanes hold the other columns of the same windows)
#pragma unroll
        for (int eh = 0; eh < 2; ++eh) {
          double v = bv[eh], sc = bs[eh];
          int xr = bi[eh] < 0 ? kNoX : xc0 + bi[eh];
#pragma unroll
          for (int m = 1; m < 4; m <<= 1) {
            const double vo = __shfl_xor_sync(0xffffffffu, v, m);
            const int xo = __shfl_xor_sync(0xffffffffu, xr, m);
            const double so = WS ? __shfl_xor_sync(0xffffffffu, sc, m) : 0.0;
            if (corr_v_better(vo, xo, v, xr)) { v = vo; xr = xo; if (WS) sc = so; }
          }
          if (t == 0) {
            const int e = (par * 4 + q) * kMWin + 16 * mi + 8 * eh + g;
            s_mv[e] = v;
            s_mx[e] = xr;
            if (WS) s_msc[e] = sc;
          }
        }
      }
      if (more) store_staged(r + 1);
    }
    __syncthreads();
    merge_row(rows_in - 1, pass);
  }
}

template <int TW, int NPL>
static CorrKernel mma_kernel(int op, bool ws, bool ssd_int) {
  if (op == kOpSsd) return ssd_int ? dense_corr_mma_kernel<TW, NPL, kOpSsdInt, false> : dense_corr_mma_kernel<TW, NPL, kOpSsd, false>;
  return ws ? dense_corr_mma_kernel<TW, NPL, kOpCorr, true> : dense_corr_mma_kernel<TW, NPL, kOpCorr, false>;
}

cudaError_t launch_corr_mma(const DevJob& J, CorrCfg cfg, int op, int np, cudaStream_t st) {
  cfg.n_xtiles = (J.nxc + kMWin - 1) / kMWin;
  cfg.n_launch_pairs = np;
  // bands: a band pays th - 1 warm-up rows (products only, about a quarter of a full row), 2 CTAs on each SM
  corr_bands(J, cfg, np, g_sm_count * 2, 0.27, J.nyc);
  const int npl = J.channels;
  const bool ws = op == kOpCorr && J.out.score != nullptr;
  const bool ssd_int = 65025ll * J.n_elems < (1ll << 28);  // u32 scoring of SSD (the sentinel of out-of-frame columns is 2^30)
  const size_t smem = (size_t)4 * npl * kMRowWords * 4 + (2 * kPassCols + 2 * kMWin) * sizeof(double2) +
                      2 * 4 * kMWin * (2 * sizeof(double) + sizeof(int));
  const CorrKernel k = J.tw > 16 ? (npl == 1 ? mma_kernel<32, 1>(op, ws, ssd_int) : mma_kernel<32, 3>(op, ws, ssd_int))
                                 : (npl == 1 ? mma_kernel<16, 1>(op, ws, ssd_int) : mma_kernel<16, 3>(op, ws, ssd_int));
  return launch_kernel(k, dim3(cfg.n_xtiles * cfg.n_bands * np), dim3(kMThreads), smem, st, J, cfg);
}

}  // namespace usv
