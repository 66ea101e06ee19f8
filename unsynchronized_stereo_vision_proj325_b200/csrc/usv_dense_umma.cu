// usv_dense_umma.cu — the correlation sweep of usv_dense_mma.cu with the row products on tcgen05 (UMMA):
// tcgen05.mma.cta_group::1.kind::i8, M = 128 windows, N = 128 or 192 candidate columns, K = 32 bytes of one plane row, u8 x u8 -> s32
// accumulators in tensor memory. Measured rate of the instruction on B200: 8 192 MAC/clk/SM, 4.2x mma.sync
// (scripts/dev/tcgen05_i8_probe.cu, which also pins the operand layout used here).
//
// Same mathematics as usv_dense_mma.cu: G_v[x, x'] = sum_c L[v][x + c] R[v][x' + c] per plane row, slid down the rows.
// UMMA reads its operands from shared memory in the canonical K-major layout (core matrices of 8 rows x 16 bytes), so
// the Toeplitz operands are materialised: row m of the A tile is the 32 bytes L[x_m .. x_m + 31] (bytes beyond the
// template width zeroed), row n of the B tile the 32 bytes R[x'_n .. x'_n + 31]; a 16-byte chunk is five aligned global
// words funnel-shifted by the byte phase. u8 x u8 products only add, so two accumulator sets live in TMEM: E = sum of G
// over every row that has entered the band so far (columns 0..191), L = sum over the rows that have left (columns
// 256..447); Sab = E - L in wrap-around u32 (the band height keeps both below 2^31). A thread of the scoring phase owns
// ONE window (its TMEM lane) and 24 of the pass's 192 columns: tcgen05.ld brings 8 accumulators of each set at a time,
// the f64 scoring is the one of usv_dense_mma.cu, there is no cross-lane reduction — four column quarters are merged
// through shared memory, passes through the global running best.
//
// Structure: no warp specialisation; per row one thread issues the 3 + 3 MMAs of the row (tiles staged during the previous
// row) and commits to an mbarrier, everybody builds the tiles of the next row in the other buffer while the tensor pipe
// works, waits (one lane per warp polls), and scores (chunks of 8 columns; chunks outside the warp's candidates are
// skipped); one __syncthreads per row. Two shapes (below): one plane — N = 128, two CTAs of 512 threads per SM; three
// planes — N = 192, one CTA of 1024 threads. The automatic dispatch (usv_dense_corr.cu) uses this kernel for one-plane
// NCC / ZNCC on frames at least 128 windows wide, where it is the fastest sweep (7.7 k pairs/s on 640x480 gray against
// 6.9 k for mma.sync); usv_set_option(USV_OPT_CORR_KERNEL, USV_CORR_KERNEL_TCGEN05) runs it wherever it applies. A
// warp-specialised version (producer / issuer / scoring warps on mbarriers) was built and measured in round 2 and is
// slower — scripts/dev/usv_dense_umma_warp_specialised_attempt.cu.txt records it and why.
#include <algorithm>
#include <cstdlib>

#include "usv_corr.cuh"

namespace usv {

// Two shapes, chosen by the number of planes (measured): one plane — N = 128, E and L take 256 TMEM columns, two CTAs of
// 512 threads per SM overlap each other's phases (7.8 k pairs/s on the 640x480 gray full-range config against 5.9 k for
// the other shape and 6.9 k for the mma.sync kernel); three planes — N = 192 in one CTA of 1 024 threads per SM (the
// tiles of three planes make the narrower pass re-stage too much: C3 2.07 k against 1.88 k).
constexpr int kUWin = 128;                 // M: windows per CTA
constexpr int kUK = 32;                    // K: bytes of one plane row per product
constexpr int kUATile = kUWin * kUK;
constexpr int u_cols(int npl) { return npl == 1 ? 128 : 192; }        // N: candidate columns per pass
constexpr int u_threads(int npl) { return npl == 1 ? 512 : 1024; }    // 4 TMEM lane groups x (threads / 128) column parts
constexpr int u_ctas(int npl) { return npl == 1 ? 2 : 1; }            // CTAs per SM (TMEM: 2 x 256 or 1 x 512 columns)
constexpr int u_tile(int npl) { return kUATile + u_cols(npl) * kUK; }
constexpr int kURawL = 176, kURawR = 256, kURaw = kURawL + kURawR;  // raw plane-row segments of one (half, plane)

__device__ __forceinline__ uint32_t u_smem(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// K-major, no swizzle; core matrix (row group rg, 16-byte K chunk kc) at (rg * 2 + kc) * 128 bytes
__device__ __forceinline__ uint64_t u_desc(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFF) >> 4) | ((uint64_t)(128 >> 4) << 16) | ((uint64_t)(256 >> 4) << 32) | ((uint64_t)1 << 46);
}
__device__ __forceinline__ void u_mma(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t}"
      ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate), "r"(0u), "r"(0u), "r"(0u), "r"(0u) : "memory");
}
__device__ __forceinline__ void u_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
                 "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
               : "r"(taddr) : "memory");
}
__device__ __forceinline__ void u_ld8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr) : "memory");
}

template <int NPL, int OP, bool WS>
__global__ void __launch_bounds__(u_threads(NPL), u_ctas(NPL)) dense_corr_umma_kernel(const DevJob J, const CorrCfg cfg) {
  constexpr int kUThreads = u_threads(NPL), kUCols = u_cols(NPL), kUNQ = kUThreads / 128, kUQCols = kUCols / kUNQ, kUTile = u_tile(NPL);
  constexpr uint32_t kUTmemCols = u_ctas(NPL) == 2 ? 256 : 512, kUAccL = kUTmemCols / 2;
  extern __shared__ __align__(1024) uint8_t usmem[];
  uint8_t* s_tiles = usmem;                                                        // [2 buffers][enter, leave][NPL][A 4 KB | B 6 KB]
  double2* s_rs = reinterpret_cast<double2*>(usmem + 4 * NPL * kUTile);            // [2][192] (Sb, rb) of the output row
  double* s_mv = reinterpret_cast<double*>(s_rs + 2 * kUCols);                     // [2][kUNQ column parts][128 windows]
  double* s_msc = s_mv + 2 * kUNQ * kUWin;
  int* s_mx = reinterpret_cast<int*>(s_msc + 2 * kUNQ * kUWin);
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_mx + 2 * kUNQ * kUWin);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bar + 1);
  uint8_t* s_raw = reinterpret_cast<uint8_t*>(s_bar) + 32;      // [2 buffers][enter, leave][NPL][L 176 B | R 256 B], 16-byte aligned

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, lg = warp & 3, cq = warp >> 2;
  const int per_tile = cfg.n_bands * cfg.n_launch_pairs;
  const int t_ord = blockIdx.x / per_tile, t_rem = blockIdx.x - t_ord * per_tile;
  const bool leftcam = J.camera_side == USV_LEFT_CAM;
  const int tile = leftcam ? cfg.n_xtiles - 1 - t_ord : t_ord;  // heaviest tiles first
  const int pair = t_rem / cfg.n_bands, band = t_rem - pair * cfg.n_bands;
  const int xm = kUWin * tile;
  const int y0 = band * cfg.bh;
  const int bh = min(cfg.bh, J.nyc - y0);
  const int th = J.th, tw = J.tw;
  const int rows_in = bh + th - 1;
  const int nxc = J.nxc;
  const uint8_t* Lb = cfg.lp + (long long)pair * cfg.pair_stride + (long long)y0 * cfg.pitch;
  const uint8_t* Rb = cfg.rp + (long long)pair * cfg.pair_stride + (long long)y0 * cfg.pitch;
  const double2* stl = cfg.stat_l + (long long)pair * J.nyc * nxc;
  const double2* str = cfg.stat_r + (long long)pair * J.nyc * nxc;
  const double nan = __longlong_as_double(0x7ff8000000000000ll);
  const double inf = __longlong_as_double(0x7ff0000000000000ll);
  const uint32_t dspan = (uint32_t)(J.dmax - J.dmin);

  int c_lo, c_hi;
  corr_cand_cols(J, leftcam, xm, kUWin, c_lo, c_hi);
  const int col_base = c_lo & ~3;
  const int n_pass = c_hi >= c_lo ? (c_hi - col_base) / kUCols + 1 : 1;

  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(u_smem(s_bar)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(u_smem(s_tmem)), "n"(kUTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t taddr = *s_tmem;
  // D = S32, A = B = unsigned 8 bit, both K-major, N = 192, M = 128
  const uint32_t idesc = (2u << 4) | ((uint32_t)(kUCols >> 3) << 17) | ((uint32_t)(kUWin >> 4) << 24);
  uint32_t bar_phase = 0;

  // scoring role of this thread: window m of the CTA (TMEM lane), column quarter cq of the pass
  const int m = 32 * lg + lane, x = xm + m;
  const uint32_t t_lane = taddr + ((uint32_t)(32 * lg) << 16);
  const double n_eff = cfg.n_eff, c0 = __dmul_rn(cfg.n_eff, -4503599627370496.0);
  const int usgn = leftcam ? -1 : 1;

  for (int pass = 0; pass < n_pass; ++pass) {
    const int xcol0 = col_base + pass * kUCols;
    const int qcol0 = xcol0 + kUQCols * cq;                       // x' of this thread's first column
    const int ub = (leftcam ? x - qcol0 : qcol0 - x) - J.dmin;    // d - dmin there; column j moves it by -/+ j
    bool first_e = true, first_l = true;                          // (thread 0) the first product of a set overwrites
    // operand tiles of the entering row r and of the leaving row r - th (a task = the two 16-byte chunks of one tile row:
    // nine aligned global words, funnel-shifted by the byte phase), statistics of the output row; buffer r & 1
    // Staging in two steps. (1) cp.async brings the raw plane-row segments a row needs (L: 160 bytes from xm, R: 224 bytes
    // from xcol0, 16-byte granules; entering and leaving row, every plane) into shared memory two rows ahead — no
    // registers, the global latency is off the critical path. (2) Thread t < 320 owns tile row t (A rows 0..127, B rows
    // 0..191) of every (half, plane): nine words of the raw segment, eight funnel shifts by the byte phase, two 16-byte
    // stores into the canonical layout. Threads 320..511 fetch the statistics of the output row.
    const int xcol0a = xcol0 & ~15;
    constexpr int kRawChunks = kURaw / 16;  // 27 per (half, plane)
    auto fetch_raw = [&](int r) {
      if (tid < 2 * NPL * kRawChunks) {
        const int hp = tid / kRawChunks, c = tid - hp * kRawChunks;
        const int half = hp / NPL, pl = hp - half * NPL;
        const int gr = r - (half ? th : 0);
        const bool is_l = c < kURawL / 16;
        const int byte0 = is_l ? xm + 16 * c : xcol0a + 16 * (c - kURawL / 16);
        if (gr >= 0 && byte0 < cfg.pitch)
          cp_async16(s_raw + ((r & 1) * 2 * NPL + hp) * kURaw + 16 * c,
                     (is_l ? Lb : Rb) + (long long)pl * cfg.plane_stride + (long long)gr * cfg.pitch + byte0);
      }
      cp_async_commit();
    };
    const bool st_on = tid < kUWin + kUCols, st_a = tid < kUWin;
    const int st_idx = st_a ? tid : tid - kUWin;
    const int st_off = st_a ? st_idx : kURawL + (xcol0 - xcol0a) + st_idx;  // first byte of the tile row in the raw segment
    const int st_w0 = st_off >> 2, st_sh = 8 * (st_off & 3);
    const int st_dst = (st_a ? 0 : kUATile) + (st_idx >> 3) * 256 + (st_idx & 7) * 16;
    auto stage = [&](int r) {
      uint8_t* tiles = s_tiles + (r & 1) * 2 * NPL * kUTile;
      if (st_on) {
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          if (r - (half ? th : 0) < 0) continue;
#pragma unroll
          for (int pl = 0; pl < NPL; ++pl) {
            const uint32_t* raw = reinterpret_cast<const uint32_t*>(s_raw + ((r & 1) * 2 * NPL + half * NPL + pl) * kURaw) + st_w0;
            uint32_t g[9];
#pragma unroll
            for (int i = 0; i < 9; ++i) g[i] = raw[i];
            uint32_t o[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) o[i] = __funnelshift_r(g[i], g[i + 1], st_sh);
            if (st_a && tw < kUK) {  // bytes of A beyond the template width are zero: K = 32 serves every width up to 32
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const int nb = tw - 4 * i;
                o[i] &= nb >= 4 ? 0xffffffffu : nb <= 0 ? 0u : (1u << (8 * nb)) - 1u;
              }
            }
            uint8_t* dst = tiles + (half * NPL + pl) * kUTile + st_dst;
            *reinterpret_cast<uint4*>(dst) = make_uint4(o[0], o[1], o[2], o[3]);
            *reinterpret_cast<uint4*>(dst + 128) = make_uint4(o[4], o[5], o[6], o[7]);
          }
        }
      } else if (r >= th - 1 && tid < kUWin + 2 * kUCols) {
        const int c = tid - (kUWin + kUCols), xk = xcol0 + c;
        s_rs[(r & 1) * kUCols + c] = xk > nxc - 1 ? make_double2(nan, nan) : __ldg(str + (long long)(y0 + r - (th - 1)) * nxc + xk);
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // the tiles are read through the async proxy
    };
    // 8-column chunks of this warp's quarter that can hold a candidate of one of its 32 windows (warp-uniform)
    uint32_t chunk_any = 0;
    {
      const int xw0 = xm + 32 * lg, xw1 = min(xw0 + 31, nxc - 1);
      for (int ch = 0; ch < kUQCols / 8; ++ch) {
        const int ca = qcol0 + 8 * ch, cb = ca + 7;
        const int d_lo = leftcam ? xw0 - cb : ca - xw1, d_hi = leftcam ? xw1 - ca : cb - xw0;
        if (xw0 <= nxc - 1 && ca <= c_hi && cb >= c_lo && d_hi >= J.dmin && d_lo <= J.dmax) chunk_any |= 1u << ch;
      }
    }
    __syncthreads();  // the previous pass is done with every buffer
    fetch_raw(0);
    if (rows_in > 1) fetch_raw(1);
    cp_async_wait_all();
    __syncthreads();
    stage(0);
    __syncthreads();
    for (int r = 0; r < rows_in; ++r) {
      const uint8_t* tiles = s_tiles + (r & 1) * 2 * NPL * kUTile;
      // the raw segments of row r + 2 into the raw buffer of row r (its tiles were built a row ago); complete and visible
      // after this row's closing barrier, i.e. before stage(r + 2)
      if (r + 2 < rows_in) fetch_raw(r + 2);
      // ---- one thread issues the products of row r: E += G_r, L += G_{r - th}
      if (tid == 0) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
        for (int pl = 0; pl < NPL; ++pl) {
          const uint32_t ta = u_smem(tiles + pl * kUTile);
          u_mma(taddr, u_desc(ta), u_desc(ta + kUATile), idesc, first_e ? 0u : 1u);
          first_e = false;
        }
        if (r >= th) {
#pragma unroll
          for (int pl = 0; pl < NPL; ++pl) {
            const uint32_t ta = u_smem(tiles + (NPL + pl) * kUTile);
            u_mma(taddr + kUAccL, u_desc(ta), u_desc(ta + kUATile), idesc, first_l ? 0u : 1u);
            first_l = false;
          }
        }
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(u_smem(s_bar)) : "memory");
      }
      // ---- while the tensor pipe works: the tiles and statistics of the next row into the other buffer (its raw
      // segments landed during the previous row), then the raw segments of the row after it into the buffer just read
      if (r + 1 < rows_in) stage(r + 1);
      // ---- everybody waits for the products: lane 0 of every warp polls. The wait is bounded by wall clock (10 s on
      // %globaltimer, far beyond any profiler or sanitizer slow-down of a microsecond-scale product); a wait that still
      // expires raises the context's status word, which the host turns into USV_ERR_CUDA, and the CTA runs on (its
      // results are then meaningless, but nothing traps and the context stays usable)
      {
        if (lane == 0) {
          uint32_t done = 0;
          const uint32_t parity = bar_phase & 1;
          unsigned long long t_start = 0;
          for (int spin = 0; !done; ++spin) {
            asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                         : "=r"(done) : "r"(u_smem(s_bar)), "r"(parity) : "memory");
            if (!done) {
              __nanosleep(64);  // the polling warps must not take the issue slots of the staging warps
              if ((spin & 1023) == 1023) {
                const unsigned long long now = global_timer_ns();
                if (t_start == 0) t_start = now;
                else if (now - t_start > 10000000000ull) { if (J.status) { *(volatile int*)J.status = kDevStatusUmmaTimeout; __threadfence_system(); } break; }
              }
            }
          }
        }
        __syncwarp();
        ++bar_phase;
      }
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      // ---- scores of the output row: this thread's window against its 48 columns, 8 at a time; the accumulators of
      // the next chunk are on their way from TMEM while the current one is scored
      if (r >= th - 1) {
        const int yo = y0 + r - (th - 1);
        const double2 La = __ldg(stl + (long long)yo * nxc + min(x, nxc - 1));
        const double2* rs = s_rs + (r & 1) * kUCols + kUQCols * cq;
        const bool has_l = r >= th;
        double bv = inf, bs = -inf;
        int bi = -1;
        const uint32_t t_col = t_lane + kUQCols * cq;
#pragma unroll
        for (int ch = 0; ch < kUQCols / 8; ++ch)
          if (chunk_any >> ch & 1) {
            uint32_t e[8], l[8];
            u_ld8(t_col + 8 * ch, e);
            if (has_l) u_ld8(t_col + kUAccL + 8 * ch, l);
            else {
#pragma unroll
              for (int i = 0; i < 8; ++i) l[i] = 0u;  // nothing has left the windows yet (the first output row of the band)
            }
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int i = 0; i < 8; ++i) {  // ascending x': a later equal candidate never replaces (P/Main.cpp:451)
              const uint32_t sab = e[i] - l[i];
              const double2 Rr = rs[8 * ch + i];
              const CorrCand c = corr_score<OP>(n_eff, c0, (int)sab, La, Rr);
              const int j = 8 * ch + i;
              if (c.v < bv && (uint32_t)(ub + usgn * j) <= dspan) { bv = c.v; bi = j; if (WS) bs = c.sc; }
            }
          }
        const int mo = ((r & 1) * kUNQ + cq) * kUWin + m;
        s_mv[mo] = bv;
        s_mx[mo] = bi < 0 ? kNoX : qcol0 + bi;
        if (WS) s_msc[mo] = bs;
      }
      cp_async_wait_all();  // the raw segments of row r + 1 (issued a row ago) are in shared memory
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncthreads();  // TMEM and this row's buffers may be overwritten; the quarters' winners are complete
      if (r >= th - 1 && tid < kUWin) {
        const int xw = xm + tid, yo = y0 + r - (th - 1), mb = (r & 1) * kUNQ * kUWin;
        double v = s_mv[mb + tid], sc = WS ? s_msc[mb + tid] : 0.0;
        int xr = s_mx[mb + tid];
#pragma unroll
        for (int qq = 1; qq < kUNQ; ++qq) {
          const double vo = s_mv[mb + qq * kUWin + tid];
          const int xo = s_mx[mb + qq * kUWin + tid];
          if (corr_v_better(vo, xo, v, xr)) { v = vo; xr = xo; if (WS) sc = s_msc[mb + qq * kUWin + tid]; }
        }
        if (xw <= nxc - 1 && corr_merge_pass<WS>(cfg, ((long long)pair * J.nyc + yo) * nxc + xw, pass, n_pass, v, xr, sc))
          corr_emit<OP>(J, cfg.pair0 + pair, xw, yo, xr, v, sc);
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kUTmemCols) : "memory");
}

template <int NPL>
static CorrKernel umma_kernel(int op, bool ws) {
  if (op == kOpSsd) return dense_corr_umma_kernel<NPL, kOpSsd, false>;
  return ws ? dense_corr_umma_kernel<NPL, kOpCorr, true> : dense_corr_umma_kernel<NPL, kOpCorr, false>;
}

cudaError_t launch_corr_umma(const DevJob& J, CorrCfg cfg, int op, int np, cudaStream_t st) {
  cfg.n_xtiles = (J.nxc + kUWin - 1) / kUWin;
  cfg.n_launch_pairs = np;
  // E and L are running sums over the rows of a band: keep them below 2^31
  const long long per_row = 65025ll * J.tw * J.channels;
  const int bh_cap = (int)std::max<long long>(1, std::min<long long>(J.nyc, ((1ll << 31) - 1) / per_row - J.th));
  corr_bands(J, cfg, np, g_sm_count * u_ctas(J.channels), 0.2, bh_cap);
  const int npl = J.channels;
  const bool ws = op == kOpCorr && J.out.score != nullptr;
  const size_t smem = (size_t)4 * npl * u_tile(npl) + 2 * u_cols(npl) * sizeof(double2) +
                      2 * (u_threads(npl) / 128) * kUWin * (2 * sizeof(double) + sizeof(int)) + 64 + (size_t)4 * npl * kURaw;
  const CorrKernel k = npl == 1 ? umma_kernel<1>(op, ws) : umma_kernel<3>(op, ws);
  return launch_kernel(k, dim3(cfg.n_xtiles * cfg.n_bands * np), dim3(u_threads(npl)), smem, st, J, cfg);
}

}  // namespace usv
