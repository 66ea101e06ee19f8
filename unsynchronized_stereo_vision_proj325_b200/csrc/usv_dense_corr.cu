// usv_dense_corr.cu — dense stride-1 sweep for the correlation costs (NCC, ZNCC), gray or interleaved colour:
// the sliding-window formulation of usv_dense.cu with IDP.4A in place of VABSDIFF4 and an exact f64 score.
// The same kernel also runs SSD (Saa + Sbb - 2 Sab from the same sums, carried as the exact f64 "score" -SSD) and SAD
// on colour frames (VABSDIFF4 per plane, "score" = -SAD); see kOpCorr / kOpSsd / kOpSad.
//
//   cost(x, x') = 1 - score,   NCC : score = (Sab * ra) * rb,            ra = 1/sqrt(Saa), rb = 1/sqrt(Sbb)
//                              ZNCC: score = ((n Sab - Sa Sb) * ra) * rb, ra = 1/sqrt(n Saa - Sa^2), rb likewise
// with every sum an exact integer over the tw x th x C window and every f64 operation the one the oracle performs
// (oracle/block_search_oracle.c:score_from_sums, usv_common.cuh:zncc_score), so scores, costs and indices are
// bit-exact. Only Sab depends on the candidate pair; the window statistics (Sa, Saa of every left window, Sb, Sbb of
// every right position) are computed once per frame by corr_stats_kernel and read back as two doubles each:
//   left  window (x, y):  (-Sa, ra)      right position (x', y):  (Sb, rb)        [NCC: (0, ra), (0, rb), n := 1]
//
// Sab slides exactly like the SAD: h(u, d, v) = sum_{b<4} L[v][u+b] * R[v][u-d+b] over the colour planes (one
// IDP.4A.U8.U8 each; interleaved frames are split into planes first, so that a packed word holds four pixels of one
// channel), V(u, d, y) = sum of h over the th rows of the window kept in a register and slid down the rows,
// Sab(x, d, y) = sum_{k < tw/4} V(x + 4k, d, y). Per candidate, v = 1 - score in f64 (usv_corr.cuh: corr_score),
// and the candidate replaces the running best iff v < best (ties: the smaller x', P/Main.cpp:451). Candidates outside
// the frame carry rb = NaN and disparities outside [search_min, search_max] carry n = NaN: their v is NaN and loses
// every comparison, so validity costs no instruction in the inner loop.
//
// Mapping: as usv_dense.cu (CTA = 4 warps = 4 byte phases, thread tile 8 positions x 4 disparities, passes of 32
// disparities, short double-fetched ring of rows per colour plane), but two CTAs per SM with up to 255 registers: the
// statistics of the row (8 windows, 11 positions) sit in registers, and the running best per window is the pair
// (score, x') in shared memory.
#include <algorithm>

#include "usv_corr.cuh"

namespace usv {

constexpr int kCThreads = 128;
constexpr int kCRB = 2;           // rows per staging block (rows are long here: a barrier every other row is cheap)
constexpr int kCLW = 32;          // words per L copy row
constexpr int kCRW = 44;          // words per R copy row (40 used)
constexpr int kCRowWords = 4 * kCLW + 4 * kCRW;
__device__ __forceinline__ uint32_t dp4a_u8(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t d;
  asm("dp4a.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}

template <int DIR, int NW, int NPL, int OP>
__device__ __forceinline__ void corr_pass(const DevJob& J, const CorrCfg& cfg, uint32_t* s_ring, double* s_bsc, int* s_bx,
                                          const uint8_t* __restrict__ Lb, const uint8_t* __restrict__ Rb, const double2* __restrict__ stl,
                                          const double2* __restrict__ str, const int X0, const int XR0, const int dbase, const int y0,
                                          const int rows_in) {
  constexpr bool SSD = OP != kOpCorr;  // integer costs: "score" = -cost, no normalisation
  const int tid = threadIdx.x, lane = tid & 31, p = tid >> 5;
  const int ul = lane & 3, dl = lane >> 2, q = dl & 3, jh = dl >> 2;
  const int th = J.th;
  const int row_words = cfg.pitch >> 2;
  const int x0 = X0 + p + 32 * ul;
  const double nan = __longlong_as_double(0x7ff8000000000000ll);

  // per disparity: n (or NaN outside [search_min, search_max]) and -n * 2^52
  double nj[4], c0j[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int d = dbase + 4 * j;
    nj[j] = (d >= J.dmin && d <= J.dmax) ? cfg.n_eff : nan;
    c0j[j] = __dmul_rn(nj[j], -4503599627370496.0);
  }
  // x' of (column i, disparity j) = xrb + 4 * k(i, j), k = i - j + 3 (LeftCam) / i + j (RightCam), k in [0, 10]
  const int xrb = DIR < 0 ? x0 - dbase - 12 : x0 + dbase;

  uint32_t V[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) V[i][j] = 0;

  // ---- staging (the short ring of usv_dense.cu, once per colour plane): slot r & 7 of the entering half and of the
  // leaving half; a task = one 16-byte chunk of one row of one plane: 5 aligned words -> 4 byte-shifted copies
  constexpr int kChunks = kCLW / 4 + 10;
  constexpr int kTasks = 2 * kCRB * NPL * kChunks;
  auto stage = [&](int row_begin) {
    for (int k = tid; k < kTasks; k += kCThreads) {
      const int half = k / (kCRB * NPL * kChunks);
      int rem = k - half * (kCRB * NPL * kChunks);
      const int rr = rem / (NPL * kChunks);
      rem -= rr * (NPL * kChunks);
      const int pl = rem / kChunks, c = rem - pl * kChunks;
      const int r = row_begin + rr, gr = r - (half ? th : 0);
      if (r >= rows_in || gr < 0) continue;
      const bool left = c < kCLW / 4;
      const int w0 = left ? 4 * c : 4 * (c - kCLW / 4);
      const uint32_t* gp = reinterpret_cast<const uint32_t*>((left ? Lb : Rb) + (long long)pl * cfg.plane_stride + (long long)gr * cfg.pitch);
      const int gb = ((left ? X0 : XR0) >> 2) + w0;
      uint32_t w[5];
#pragma unroll
      for (int t = 0; t < 5; ++t) w[t] = __ldg(gp + min(max(gb + t, 0), row_words - 1));
      const int kw = left ? kCLW : kCRW;
      uint32_t* dst = s_ring + ((size_t)((half * 2 * kCRB + (r & (2 * kCRB - 1))) * NPL + pl)) * kCRowWords + (left ? 0 : 4 * kCLW) + w0;
      *reinterpret_cast<uint4*>(dst) = make_uint4(w[0], w[1], w[2], w[3]);
#pragma unroll
      for (int s = 1; s < 4; ++s)
        *reinterpret_cast<uint4*>(dst + s * kw) = make_uint4(__funnelshift_r(w[0], w[1], 8 * s), __funnelshift_r(w[1], w[2], 8 * s),
                                                             __funnelshift_r(w[2], w[3], 8 * s), __funnelshift_r(w[3], w[4], 8 * s));
    }
  };

  const uint32_t* my_l = s_ring + p * kCLW + 8 * ul;
  const uint32_t* my_r = s_ring + 4 * kCLW + q * kCRW + 8 * ul + (DIR < 0 ? 4 - 4 * jh : 4 * jh);
  const int own_i = ((dl >> 2) & 1) * 4 + ((dl >> 1) & 1) * 2 + (dl & 1);
  const bool b4 = (dl >> 2) & 1, b3 = (dl >> 1) & 1, b2 = dl & 1;
  const int my_pos = p * 32 + 8 * ul + own_i;

  auto row_body = [&](auto has_old_t, auto has_keys_t, int row) {
    constexpr bool HAS_OLD = decltype(has_old_t)::value, HAS_KEYS = decltype(has_keys_t)::value;
    const int slot = row & (2 * kCRB - 1);
#pragma unroll
    for (int pl = 0; pl < NPL; ++pl) {
      {
        const uint4* lp = reinterpret_cast<const uint4*>(my_l + (size_t)(slot * NPL + pl) * kCRowWords);
        const uint4* rp = reinterpret_cast<const uint4*>(my_r + (size_t)(slot * NPL + pl) * kCRowWords);
        const uint4 l0 = lp[0], l1 = lp[1], r0 = rp[0], r1 = rp[1], r2 = rp[2];
        const uint32_t Lw[8] = {l0.x, l0.y, l0.z, l0.w, l1.x, l1.y, l1.z, l1.w};
        const uint32_t Rw[12] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w, r2.x, r2.y, r2.z, r2.w};
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const uint32_t rw = Rw[DIR < 0 ? i - j + 4 : i + j];
            V[i][j] = OP == kOpSad ? sad4_acc(Lw[i], rw, V[i][j]) : dp4a_u8(Lw[i], rw, V[i][j]);
          }
      }
      if (HAS_OLD) {
        const uint4* lo = reinterpret_cast<const uint4*>(my_l + (size_t)((2 * kCRB + slot) * NPL + pl) * kCRowWords);
        const uint4* ro = reinterpret_cast<const uint4*>(my_r + (size_t)((2 * kCRB + slot) * NPL + pl) * kCRowWords);
        const uint4 m0 = lo[0], m1 = lo[1], s0 = ro[0], s1 = ro[1], s2 = ro[2];
        const uint32_t Lw[8] = {m0.x, m0.y, m0.z, m0.w, m1.x, m1.y, m1.z, m1.w};
        const uint32_t Rw[12] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w, s2.x, s2.y, s2.z, s2.w};
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const uint32_t rw = Rw[DIR < 0 ? i - j + 4 : i + j];
            V[i][j] -= OP == kOpSad ? sad4_acc(Lw[i], rw, 0u) : dp4a_u8(Lw[i], rw, 0u);
          }
      }
    }
    if (HAS_KEYS) {
      const int yo = y0 + row - (th - 1);  // output row
      // statistics of the row: this thread's 8 windows and the 11 right positions its 32 candidates touch
      const double2* ls = stl + (long long)yo * J.nxc;
      const double2* rs = str + (long long)yo * J.nxc;
      double2 La[8], Rs[11];
#pragma unroll
      for (int i = 0; i < 8; ++i) La[i] = __ldg(ls + min(max(x0 + 4 * i, 0), J.nxc - 1));
#pragma unroll
      for (int k = 0; k < 11; ++k) {
        const int xk = xrb + 4 * k;
        Rs[k] = __ldg(rs + min(max(xk, 0), J.nxc - 1));
        if (xk < 0 || xk > J.nxc - 1) { Rs[k].y = nan; if (SSD) Rs[k].x = nan; }  // a candidate outside the frame loses every comparison
      }
      // halo columns 8 .. 8+NW-2 from the next u-lane; window sums of column 0
      uint32_t Hx[NW - 1][4], T[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
#pragma unroll
        for (int c = 0; c < NW - 1; ++c) Hx[c][j] = __shfl_down_sync(0xffffffffu, V[c][j], 1, 4);
        uint32_t t = 0;
#pragma unroll
        for (int k = 0; k < NW; ++k) t += k < 8 ? V[k][j] : Hx[k - 8][j];
        T[j] = t;
      }
      double bsc[8];
      int bx[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        double best_v = __longlong_as_double(0x7ff0000000000000ll), best_sc = __longlong_as_double(0xfff0000000000000ll);
        int best_x = kNoX;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int k = DIR < 0 ? i - j + 3 : i + j;
          const CorrCand c = corr_score<OP>(nj[j], c0j[j], (int)T[j], La[i], Rs[k]);
          // j ascending = x' descending (LeftCam) / ascending (RightCam): on a tie the smaller x' stays
          const bool take = DIR < 0 ? c.v <= best_v : c.v < best_v;
          if (take) { best_v = c.v; best_sc = c.sc; best_x = xrb + 4 * k; }
          if (i < 7) T[j] += (i + NW < 8 ? V[i + NW][j] : Hx[i + NW - 8][j]) - V[i][j];
        }
        bsc[i] = best_sc; bx[i] = best_x;
      }
      // reduce-scatter over the 8 d-lanes (lane bits 4, 3, 2): each lane ends with the best of one window
      double h4s[4], h2s[2], h1s;
      int h4x[4], h2x[2], h1x;
      auto merge = [&](double& sc_m, int& x_m, double sc_send, int x_send, int lane_mask) {
        const double sc_o = __shfl_xor_sync(0xffffffffu, sc_send, lane_mask);
        const int x_o = __shfl_xor_sync(0xffffffffu, x_send, lane_mask);
        if (corr_better(sc_o, x_o, sc_m, x_m)) { sc_m = sc_o; x_m = x_o; }
      };
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        h4s[k] = b4 ? bsc[4 + k] : bsc[k]; h4x[k] = b4 ? bx[4 + k] : bx[k];
        merge(h4s[k], h4x[k], b4 ? bsc[k] : bsc[4 + k], b4 ? bx[k] : bx[4 + k], 16);
      }
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        h2s[k] = b3 ? h4s[2 + k] : h4s[k]; h2x[k] = b3 ? h4x[2 + k] : h4x[k];
        merge(h2s[k], h2x[k], b3 ? h4s[k] : h4s[2 + k], b3 ? h4x[k] : h4x[2 + k], 8);
      }
      h1s = b2 ? h2s[1] : h2s[0]; h1x = b2 ? h2x[1] : h2x[0];
      merge(h1s, h1x, b2 ? h2s[0] : h2s[1], b2 ? h2x[0] : h2x[1], 4);
      const int e = (row - (th - 1)) * 128 + my_pos;
      if (corr_better(h1s, h1x, s_bsc[e], s_bx[e])) { s_bsc[e] = h1s; s_bx[e] = h1x; }
    }
  };
  auto block_edge = [&](int row) {
    if ((row & (kCRB - 1)) == 0) {
      __syncthreads();
      stage(row + kCRB);
    }
  };

  __syncthreads();
  stage(0);
  int row = 0;
  const int warm = min(th - 1, rows_in);
  for (; row < warm; ++row) {
    block_edge(row);
    row_body(std::false_type{}, std::false_type{}, row);
  }
  if (row < rows_in) {
    block_edge(row);
    row_body(std::false_type{}, std::true_type{}, row);
    ++row;
  }
  for (; row < rows_in; ++row) {
    block_edge(row);
    row_body(std::true_type{}, std::true_type{}, row);
  }
}

template <int DIR, int NW, int NPL, int OP>
__global__ void __launch_bounds__(kCThreads, 3) dense_corr_argmin_kernel(const DevJob J, const CorrCfg cfg) {
  extern __shared__ __align__(16) uint32_t smem_u32[];
  uint32_t* s_ring = smem_u32;                                              // [2][2*kCRB][NPL][kCRowWords]
  double* s_bsc = reinterpret_cast<double*>(smem_u32 + 4 * kCRB * NPL * kCRowWords);  // [bh][128] best score
  int* s_bx = reinterpret_cast<int*>(s_bsc + (size_t)cfg.bh * 128);                  // [bh][128] its x'

  const int tid = threadIdx.x, lane = tid & 31, p = tid >> 5;
  const int dl = lane >> 2;
  const int tile = blockIdx.x, band = blockIdx.y, pair = blockIdx.z;
  const int X0 = tile * cfg.stride_px - cfg.x_off;
  const int y0 = band * cfg.bh;
  const int bh = min(cfg.bh, J.nyc - y0);
  const int rows_in = bh + J.th - 1;
  const uint8_t* Lb = cfg.lp + (long long)pair * cfg.pair_stride + (long long)y0 * cfg.pitch;
  const uint8_t* Rb = cfg.rp + (long long)pair * cfg.pair_stride + (long long)y0 * cfg.pitch;
  const double2* stl = cfg.stat_l + (long long)pair * J.nyc * J.nxc;
  const double2* str = cfg.stat_r + (long long)pair * J.nyc * J.nxc;

  for (int i = tid; i < bh * 128; i += kCThreads) { s_bsc[i] = __longlong_as_double(0xfff0000000000000ll); s_bx[i] = kNoX; }

  const int x_lo = max(X0, 0), x_hi = min(X0 + cfg.stride_px - 1, J.nxc - 1);
  int d_lo, d_hi;
  if (DIR < 0) { d_lo = max(J.dmin, x_lo - (J.nxc - 1)); d_hi = min(J.dmax, x_hi); }
  else { d_lo = max(J.dmin, -x_hi); d_hi = min(J.dmax, J.nxc - 1 - x_lo); }
  d_lo = d_lo & ~3;
  const int n_pass = d_hi >= d_lo ? (d_hi - d_lo + 3) / 32 + 1 : 0;
  for (int pass = 0; pass < n_pass; ++pass) {
    const int D0 = d_lo + 32 * pass;
    const int dbase = D0 + 16 * (dl >> 2) + (DIR < 0 ? (p - (dl & 3)) : ((dl & 3) - p));
    const int XR0 = DIR < 0 ? X0 - D0 - 32 : X0 + D0;
    corr_pass<DIR, NW, NPL, OP>(J, cfg, s_ring, s_bsc, s_bx, Lb, Rb, stl, str, X0, XR0, dbase, y0, rows_in);
  }
  __syncthreads();

  // ---- fused epilogue: (score, x') -> Match / disparity / distance
  const int n_pos = 32 - NW + 1;
  const int span = min(cfg.stride_px, J.nxc - X0);
  for (int idx = tid; idx < bh * span; idx += kCThreads) {
    const int yy = idx / span, xo = idx - yy * span;
    const int pp = xo & 3, a = xo >> 2;
    if (a >= n_pos || X0 + xo < 0) continue;
    const int e = (yy * 4 + pp) * 32 + a;
    const double sc = s_bsc[e];
    corr_emit<OP>(J, cfg.pair0 + pair, X0 + xo, y0 + yy, s_bx[e], __dsub_rn(1.0, sc), sc);
  }
}

// ---- per-frame preparation -------------------------------------------------------------------------------------
// interleaved [H][row_stride] (C channels) -> planes [C][H][pitch]
__global__ void corr_planes_kernel(const uint8_t* __restrict__ src, long long src_frame_stride, int row_stride, int width, int height,
                                   int channels, uint8_t* __restrict__ dst, long long dst_pair_stride, long long plane_stride, int pitch) {
  const int pair = blockIdx.z, y = blockIdx.y;
  const uint8_t* s = src + (long long)pair * src_frame_stride + (long long)y * row_stride;
  uint8_t* d = dst + (long long)pair * dst_pair_stride + (long long)y * pitch;
  for (int x = blockIdx.x * blockDim.x + threadIdx.x; x < pitch; x += gridDim.x * blockDim.x)
    for (int c = 0; c < channels; ++c) d[(long long)c * plane_stride + x] = x < width ? s[x * channels + c] : 0;
}

// Window statistics of one camera in two sliding stages (a few loads per window instead of 2 * tw * C):
//   corr_rowsum_kernel  rs[y][x] = (sum, sum of squares) of the tw * C bytes of row y starting at pixel x; a thread
//                       owns a run of 32 consecutive x of one row and slides: + the C bytes entering, - the C leaving
//   corr_stats_kernel   vertical sliding sum of th rows of rs -> (left ? -Sa : Sb, 1/sqrt(variance term)) with the
//                       oracle's operations (usv_common.cuh ncc_score / zncc_score); thread = (x, band of rows)
__global__ void corr_rowsum_kernel(const uint8_t* __restrict__ frames, long long frame_stride, int row_stride, int channels, int tw,
                                   int nxc, int height, uint2* __restrict__ rs) {
  const int run = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y, pair = blockIdx.z;
  const int xa = run * 32;
  if (xa >= nxc) return;
  const int xb = min(xa + 32, nxc);
  const uint8_t* r = frames + (long long)pair * frame_stride + (long long)y * row_stride;
  const int nb = tw * channels;
  uint32_t s1 = 0, s2 = 0;
  for (int k = 0; k < nb; ++k) { const uint32_t v = __ldg(r + xa * channels + k); s1 += v; s2 += v * v; }
  uint2* o = rs + ((long long)pair * height + y) * nxc;
  for (int x = xa; x < xb; ++x) {
    o[x] = make_uint2(s1, s2);
    if (x + 1 < xb)
      for (int c = 0; c < channels; ++c) {
        const uint32_t vin = __ldg(r + (x + tw) * channels + c), vout = __ldg(r + x * channels + c);
        s1 += vin - vout; s2 += vin * vin - vout * vout;
      }
  }
}

// The same row sums by prefix sums, one block per frame row: the row is read once with coalesced word loads (each thread
// keeps its kScanWords words in registers), (sum, sum of squares) are scanned over the block, the exclusive prefix at every
// pixel boundary goes to shared memory, and rs[y][x] = prefix[x + tw] - prefix[x] is written coalesced. Exact integers
// (u32: a row of 8 192 bytes sums to < 2^30). Used when the row fits kScanThreads * kScanWords words.
constexpr int kScanThreads = 256, kScanWords = 8;
__global__ void __launch_bounds__(kScanThreads) corr_rowsum_scan_kernel(const uint8_t* __restrict__ frames, long long frame_stride, int row_stride,
                                                                        int channels, int tw, int nxc, int width, int height, uint2* __restrict__ rs) {
  extern __shared__ uint2 s_ps[];  // [width + 1]
  __shared__ uint2 s_warp[kScanThreads / 32];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int y = blockIdx.x, pair = blockIdx.y;
  const int nb = width * channels, nwords = (nb + 3) >> 2;
  const int K = (nwords + kScanThreads - 1) / kScanThreads;  // words per thread (<= kScanWords, checked on the host)
  const uint32_t* row = reinterpret_cast<const uint32_t*>(frames + (long long)pair * frame_stride + (long long)y * row_stride);
  const int w0 = tid * K;
  uint32_t wv[kScanWords];
  uint32_t s1 = 0, s2 = 0;
#pragma unroll
  for (int k = 0; k < kScanWords; ++k) {
    uint32_t w = 0;
    if (k < K && w0 + k < nwords) {
      w = __ldg(row + w0 + k);
      const int left = nb - 4 * (w0 + k);  // bytes of this word inside the row
      if (left < 4) w &= (1u << (8 * left)) - 1u;
    }
    wv[k] = w;
    s1 = dp4a_u8(w, 0x01010101u, s1);
    s2 = dp4a_u8(w, w, s2);
  }
  // exclusive block scan of the per-thread totals
  uint32_t i1 = s1, i2 = s2;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t a = __shfl_up_sync(0xffffffffu, i1, o), b = __shfl_up_sync(0xffffffffu, i2, o);
    if (lane >= o) { i1 += a; i2 += b; }
  }
  if (lane == 31) s_warp[wid] = make_uint2(i1, i2);
  __syncthreads();
  uint32_t p1 = i1 - s1, p2 = i2 - s2;
  for (int k = 0; k < wid; ++k) { p1 += s_warp[k].x; p2 += s_warp[k].y; }
  // walk the thread's bytes: the running prefix at every pixel boundary (also the one that closes the chunk; the next
  // thread writes the same value there)
  int b = 4 * w0;
  int ph = b % channels, px = b / channels;  // byte b = channel ph of pixel px
#pragma unroll
  for (int k = 0; k < kScanWords; ++k) {
    if (k < K) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if (ph == 0 && px <= width) s_ps[px] = make_uint2(p1, p2);
        const uint32_t v = (wv[k] >> (8 * i)) & 0xffu;
        p1 += v; p2 += v * v;
        if (++ph == channels) { ph = 0; ++px; }
      }
    }
  }
  if (ph == 0 && px <= width) s_ps[px] = make_uint2(p1, p2);
  __syncthreads();
  uint2* o = rs + ((long long)pair * height + y) * nxc;
  for (int x = tid; x < nxc; x += kScanThreads) {
    const uint2 hi = s_ps[x + tw], lo = s_ps[x];
    o[x] = make_uint2(hi.x - lo.x, hi.y - lo.y);
  }
}

__global__ void corr_stats_kernel(const uint2* __restrict__ rs, int height, int tw, int th, int channels, int nxc, int nyc, int kind,
                                  int is_left, int band_rows, double2* __restrict__ out) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int pair = blockIdx.z;
  if (x >= nxc) return;
  const int y0 = blockIdx.y * band_rows, y1 = min(y0 + band_rows, nyc);
  const uint2* col = rs + (long long)pair * height * nxc + x;
  const long long n = (long long)tw * th * channels;
  long long sa = 0, saa = 0;
#pragma unroll 8
  for (int v = 0; v < th - 1; ++v) { const uint2 q = __ldg(col + (long long)(y0 + v) * nxc); sa += q.x; saa += q.y; }
#pragma unroll 4
  for (int y = y0; y < y1; ++y) {
    const uint2 qin = __ldg(col + (long long)(y + th - 1) * nxc);
    sa += qin.x; saa += qin.y;
    double m, r;
    if (kind == USV_COST_SAD) {
      m = 0.0;  // score = -SAD
      r = 1.0;
    } else if (kind == USV_COST_SSD) {
      m = -(double)saa;  // both cameras: score = 2 Sab - Saa - Sbb
      r = 1.0;
    } else if (kind == USV_COST_NCC) {
      m = 0.0;
      r = saa == 0 ? 0.0 : __drcp_rn(__dsqrt_rn((double)saa));
    } else {
      const long long da = n * saa - sa * sa;
      m = is_left ? -(double)sa : (double)sa;
      r = da == 0 ? 0.0 : __drcp_rn(__dsqrt_rn((double)da));
    }
    out[((long long)pair * nyc + y) * nxc + x] = make_double2(m, r);
    const uint2 qout = __ldg(col + (long long)y * nxc);
    sa -= qout.x; saa -= qout.y;
  }
}

// colour planes of both cameras for the sweep below and for the colour SAD sweep of usv_dense.cu (kernels are launched
// from the translation unit that defines them)
cudaError_t launch_split_planes(const DevJob& J, int pair0, int np, uint8_t* dst_l, uint8_t* dst_r, int pitch, cudaStream_t st) {
  const long long plane_stride = (long long)J.height * pitch, pair_stride = plane_stride * J.channels;
  const dim3 g((pitch + 255) / 256, J.height, np);
  corr_planes_kernel<<<g, 256, 0, st>>>(J.left + (long long)pair0 * J.frame_stride, J.frame_stride, J.row_stride, J.width, J.height, J.channels, dst_l,
                                        pair_stride, plane_stride, pitch);
  corr_planes_kernel<<<g, 256, 0, st>>>(J.right + (long long)pair0 * J.frame_stride, J.frame_stride, J.row_stride, J.width, J.height, J.channels, dst_r,
                                        pair_stride, plane_stride, pitch);
  return cudaGetLastError();
}

// Pair scratch of launch_dense_corr for a chunk of np pairs: the colour planes of both cameras (colour frames only);
// 256-byte aligned, the window statistics of both cameras and the row sums they are made from; 256-byte aligned, the
// tensor-pipe sweeps' running best (v, score, x'). per_pair sets the chunk sizes. Its 1 280 bytes of slack cover the two
// alignments (at most 510 bytes a chunk), so np * per_pair bytes hold a chunk of np pairs.
struct CorrScratch {
  size_t per_pair;
  size_t planes_r, stat_l, stat_r, rsum, best_v, best_sc, best_x;  // offsets inside the chunk (left planes at 0)
};
static CorrScratch corr_scratch(const DevJob& J, size_t np) {
  const size_t planes = J.channels > 1 ? (size_t)J.channels * J.height * colour_plane_pitch(J) : 0;  // of one camera
  const size_t win = (size_t)J.nyc * J.nxc, rows = (size_t)J.height * J.nxc;
  auto align = [](size_t b) { return (b + 255) & ~(size_t)255; };
  CorrScratch s;
  s.per_pair = 2 * planes + 2 * win * sizeof(double2) + rows * sizeof(uint2) + win * (2 * sizeof(double) + sizeof(int)) + 1280;
  s.planes_r = np * planes;
  s.stat_l = align(2 * np * planes);
  s.stat_r = s.stat_l + np * win * sizeof(double2);
  s.rsum = s.stat_r + np * win * sizeof(double2);
  s.best_v = align(s.rsum + np * rows * sizeof(uint2));
  s.best_sc = s.best_v + np * win * sizeof(double);
  s.best_x = s.best_sc + np * win * sizeof(double);
  return s;
}

size_t corr_scratch_bytes_per_pair(const DevJob& J) { return corr_scratch(J, 1).per_pair; }

// coverage of both tensor-pipe sweeps
static bool corr_tensor_supported(const DevJob& J, int op) {
  if (op == kOpSad) return false;               // |a - b| is not a product
  if (J.tw < 1 || J.tw > 32) return false;      // K = 32 bytes of one product; narrower templates zero the unused bytes of A
  return 255ll * 255 * J.n_elems < (1ll << 31);  // Sab must fit the s32 accumulators
}

void corr_bands(const DevJob& J, CorrCfg& cfg, int np, int slots, double warm_weight, int bh_cap) {
  double best_eff = -1.0;
  int best_nb = (J.nyc + bh_cap - 1) / bh_cap;
  for (int nb = best_nb; nb <= std::max(best_nb, J.nyc / 8); ++nb) {
    const int bh = (J.nyc + nb - 1) / nb, nbb = (J.nyc + bh - 1) / bh;
    if (bh > bh_cap) continue;
    const long long ctas = (long long)nbb * cfg.n_xtiles * np;
    const long long waves = (ctas + slots - 1) / slots;
    const double eff = (double)ctas / (double)(waves * slots) * bh / (bh + warm_weight * (J.th - 1));
    if (eff > best_eff * 1.005) { best_eff = eff; best_nb = nbb; }
  }
  cfg.bh = (J.nyc + best_nb - 1) / best_nb;
  cfg.n_bands = (J.nyc + cfg.bh - 1) / cfg.bh;
}

template <int DIR, int NW, int NPL>
static CorrKernel alu_kernel_op(int op) {
  return op == kOpSsd ? dense_corr_argmin_kernel<DIR, NW, NPL, kOpSsd>
       : op == kOpSad ? dense_corr_argmin_kernel<DIR, NW, NPL, kOpSad>
                      : dense_corr_argmin_kernel<DIR, NW, NPL, kOpCorr>;
}
template <int DIR, int NPL>
static CorrKernel alu_kernel(int nw, int op) {
  switch (nw) {
    case 2: return alu_kernel_op<DIR, 2, NPL>(op);
    case 3: return alu_kernel_op<DIR, 3, NPL>(op);
    case 4: return alu_kernel_op<DIR, 4, NPL>(op);
    case 6: return alu_kernel_op<DIR, 6, NPL>(op);
    default: return alu_kernel_op<DIR, 8, NPL>(op);
  }
}

constexpr size_t kCSmemBudget = 74 * 1024;  // three CTAs per SM
static_assert((kCSmemBudget - (size_t)4 * kCRB * 3 * kCRowWords * 4) / (128 * 12) >= 8, "bands of at least 8 rows");

// The ALU sweep: x-tiles of 4 * (33 - tw / 4) windows; as many bands as shared memory requires, more while the grid of
// the whole batch (n_pairs) fills fewer than two CTAs per SM
static cudaError_t launch_corr_alu(const DevJob& J, CorrCfg cfg, int op, int np, int n_pairs, cudaStream_t st) {
  const int nw = J.tw / 4, npl = J.channels;
  cfg.stride_px = 4 * (32 - nw + 1);
  cfg.n_xtiles = (J.nxc + cfg.stride_px - 1) / cfg.stride_px;
  cfg.x_off = J.camera_side == USV_LEFT_CAM ? ((cfg.n_xtiles * cfg.stride_px - J.nxc) & ~3) : 0;
  const size_t ring_bytes = (size_t)4 * kCRB * npl * kCRowWords * 4;
  const int bh_max = (int)((kCSmemBudget - ring_bytes) / (128 * 12));
  int n_bands = (J.nyc + bh_max - 1) / bh_max;
  while ((long long)n_bands * cfg.n_xtiles * n_pairs < g_sm_count * 2 && n_bands < (J.nyc + 15) / 16) ++n_bands;
  cfg.bh = (J.nyc + n_bands - 1) / n_bands;
  cfg.n_bands = (J.nyc + cfg.bh - 1) / cfg.bh;
  const size_t smem = ring_bytes + (size_t)cfg.bh * 128 * 12;
  const CorrKernel k = J.camera_side == USV_LEFT_CAM ? (npl == 1 ? alu_kernel<-1, 1>(nw, op) : alu_kernel<-1, 3>(nw, op))
                                                     : (npl == 1 ? alu_kernel<1, 1>(nw, op) : alu_kernel<1, 3>(nw, op));
  return launch_corr_kernel(k, dim3(cfg.n_xtiles, cfg.n_bands, np), dim3(kCThreads), smem, st, J, cfg);
}

// Returns cudaErrorNotSupported when the job is outside the coverage of the three sweeps (the caller then runs the
// direct form).
cudaError_t launch_dense_corr(const DevJob& J, int n_pairs, void* d_scratch, size_t scratch_bytes, cudaStream_t st, const char** kernel_name,
                              int* n_launches) {
  *n_launches = 0;
  if (J.tx || J.sx != 1 || J.sy != 1) return cudaErrorNotSupported;
  if (J.cost_kind != USV_COST_NCC && J.cost_kind != USV_COST_ZNCC && J.cost_kind != USV_COST_SSD && J.cost_kind != USV_COST_SAD)
    return cudaErrorNotSupported;
  if (J.channels != 1 && J.channels != 3) return cudaErrorNotSupported;
  if (J.cost_rows || J.score_rows) return cudaErrorNotSupported;
  const int op = J.cost_kind == USV_COST_SSD ? kOpSsd : J.cost_kind == USV_COST_SAD ? kOpSad : kOpCorr;
  // the sweep: a tensor-pipe kernel wherever one covers the job (any width up to 32, any height, not SAD): tcgen05 for
  // one-plane NCC / ZNCC on frames at least 128 windows wide, mma.sync otherwise; else the ALU kernel (widths
  // 8 / 12 / 16 / 24 / 32, th <= 64). J.corr_kernel (usv_set_option USV_OPT_CORR_KERNEL, a test / measurement aid):
  // 0 = this choice, otherwise the named sweep wherever it covers the job
  const int nw = J.tw / 4;
  const bool alu_ok = J.tw % 4 == 0 && (nw == 2 || nw == 3 || nw == 4 || nw == 6 || nw == 8) && J.th <= 64 &&
                      255ll * 255 * J.n_elems < (1ll << 32);  // Sab must fit the u32 accumulators
  const bool tensor_ok = J.corr_kernel != USV_CORR_KERNEL_ALU && corr_tensor_supported(J, op);
  if (!alu_ok && !tensor_ok) return cudaErrorNotSupported;
  const bool umma = J.corr_kernel == USV_CORR_KERNEL_TCGEN05 ||
                    (J.corr_kernel == USV_CORR_KERNEL_AUTO && J.channels == 1 && op == kOpCorr && J.nxc >= 128);
  enum Sweep { kAlu, kMma, kUmma };
  const Sweep sweep = !tensor_ok ? kAlu : umma ? kUmma : kMma;

  const size_t per_pair = corr_scratch_bytes_per_pair(J);
  if (scratch_bytes < per_pair) return cudaErrorNotSupported;
  const int chunk = (int)std::min<size_t>((size_t)n_pairs, scratch_bytes / per_pair);

  CorrCfg cfg = {};
  cfg.n_eff = J.cost_kind == USV_COST_ZNCC ? (double)J.n_elems : J.cost_kind == USV_COST_SSD ? 2.0 : J.cost_kind == USV_COST_SAD ? -1.0 : 1.0;
  for (int p0 = 0; p0 < n_pairs; p0 += chunk) {
    const int np = std::min(chunk, n_pairs - p0);
    const CorrScratch s = corr_scratch(J, np);
    uint8_t* const base = (uint8_t*)d_scratch;  // 256-byte aligned (cudaMalloc)
    cfg.pair0 = p0;
    if (J.channels > 1) {
      cfg.pitch = colour_plane_pitch(J);
      cfg.plane_stride = (long long)J.height * cfg.pitch;
      cfg.pair_stride = cfg.plane_stride * J.channels;
      cfg.lp = base;
      cfg.rp = base + s.planes_r;
      const cudaError_t e = launch_split_planes(J, p0, np, base, base + s.planes_r, cfg.pitch, st);
      if (e != cudaSuccess) return e;
      *n_launches += 2;
    } else {
      cfg.lp = J.left + (long long)p0 * J.frame_stride;
      cfg.rp = J.right + (long long)p0 * J.frame_stride;
      cfg.pitch = J.row_stride; cfg.plane_stride = 0; cfg.pair_stride = J.frame_stride;
    }
    // window statistics of each camera: row sums into rsum ([np][H][nxc], by prefix sums when the row fits one block's
    // registers, else sliding), then their vertical sliding sums
    uint2* rsum = (uint2*)(base + s.rsum);
    double2* stat[2] = {(double2*)(base + s.stat_l), (double2*)(base + s.stat_r)};
    const int band_rows = 32;  // short bands: the kernel is latency-bound (one dependent load chain per thread)
    const dim3 g1(((J.nxc + 31) / 32 + 63) / 64, J.height, np);
    const dim3 g2((J.nxc + 127) / 128, (J.nyc + band_rows - 1) / band_rows, np);
    const bool scan = (J.width * J.channels + 3) / 4 <= kScanThreads * kScanWords;
    const dim3 gs(J.height, np);
    const size_t smem_scan = (size_t)(J.width + 1) * sizeof(uint2);
    for (int cam = 0; cam < 2; ++cam) {
      const uint8_t* f = (cam ? J.right : J.left) + (long long)p0 * J.frame_stride;
      if (scan) corr_rowsum_scan_kernel<<<gs, kScanThreads, smem_scan, st>>>(f, J.frame_stride, J.row_stride, J.channels, J.tw, J.nxc, J.width, J.height, rsum);
      else corr_rowsum_kernel<<<g1, 64, 0, st>>>(f, J.frame_stride, J.row_stride, J.channels, J.tw, J.nxc, J.height, rsum);
      corr_stats_kernel<<<g2, 128, 0, st>>>(rsum, J.height, J.tw, J.th, J.channels, J.nxc, J.nyc, J.cost_kind, cam == 0, band_rows, stat[cam]);
    }
    *n_launches += 4;
    cfg.stat_l = stat[0];
    cfg.stat_r = stat[1];
    cfg.best_v = (double*)(base + s.best_v);
    cfg.best_sc = (double*)(base + s.best_sc);
    cfg.best_x = (int*)(base + s.best_x);
    const cudaError_t e = sweep == kAlu   ? launch_corr_alu(J, cfg, op, np, n_pairs, st)
                          : sweep == kMma ? launch_corr_mma(J, cfg, op, np, st)
                                          : launch_corr_umma(J, cfg, op, np, st);
    if (e != cudaSuccess) return e;
    *n_launches += 1;
  }
  *kernel_name = sweep == kAlu ? "dense_corr_argmin_kernel" : sweep == kMma ? "dense_corr_mma_kernel" : "dense_corr_umma_kernel";
  return cudaSuccess;
}

}  // namespace usv
