// usv_dense_kernel.cuh — the sliding-window SAD kernel templates (described in usv_dense.cu) and the choice of the kernel
// of one (planes, disparities per thread, cost) variant. Included by the translation units that instantiate the variants
// (usv_dense.cu: gray JT = 4, usv_dense_g8.cu: gray JT = 8, usv_dense_colour.cu: three planes; usv_dense_census.cu and
// usv_dense_census_colour.cu: the same for census frames) so that they compile in parallel; nothing here is specific to
// one of them.
//
// CENSUS: the Hamming arm. The frames are census frames (usv_census.cu) and a packed word of four bytes costs
// popc(a ^ b) (LOP3 + POPC) instead of sum |a - b| (VABSDIFF4); everything else (ring, byte-shifted copies, sliding V
// sums, keys, BIG columns, fold, thin pass, epilogue) is the same code.
#pragma once
#include <algorithm>
#include <type_traits>

#include "usv_common.cuh"

namespace usv {

constexpr int kDenseThreads = 128;
constexpr int kLW = 32;         // words per L copy row (128 B)
// JT = disparities per thread of a regular pass (4: 32 per warp; 8: 64 per warp, the colour sweep — twice the VABSDIFF4 per
// shared-memory operand word). Words per R copy row: 24 + 2 JT + 8 used (40 / 48); 44 / 52 keep the four copies on disjoint banks.
constexpr int r_copy_words(int jt) { return jt == 4 ? 44 : 52; }
constexpr int r_copy_chunks(int jt) { return (32 + 2 * jt) / 4; }   // 16-byte chunks of the R segment staged per row: 10 / 12
constexpr int row_words(int jt) { return 4 * kLW + 4 * r_copy_words(jt); }  // one ring row: 4 L copies + 4 R copies
constexpr int kCodeOff = 32;    // candidate code = x0 -/+ d + kCodeOff: a valid candidate of column i has x0 -/+ d >= -4i >= -28

struct DenseCfg {
  int stride_px;    // x-tile stride = 4 * (32 - tw/4 + 1)
  int n_xtiles;
  int bh;           // output rows per band
  int n_bands;
  int xb;           // bits of the candidate code inside the key
  int ring_words;   // shared-memory words of the row ring
  int x_off;        // tile t starts at x = t * stride_px - x_off (multiple of 4)
  int n_pairs;      // the grid is one-dimensional: chunks of pairs, inside a chunk tile-major, heaviest tiles first
  int chunk_pairs;
  // where the rows come from: the frames themselves (one plane) or the planes buffer [pair][plane][H][pitch] the
  // interleaved colour frames were split into (usv_dense_corr.cu: corr_planes_kernel)
  const uint8_t* lp;
  const uint8_t* rp;
  long long pair_stride, plane_stride;
  int pitch;        // bytes between rows of a plane
  int pair0;        // first pair of this launch inside the caller's batch (outputs are indexed by the global pair)
};

// c + the cost of four packed bytes of the sweep's cost
template <bool CENSUS>
__device__ __forceinline__ uint32_t cost4_acc(uint32_t a, uint32_t b, uint32_t c) {
  if constexpr (CENSUS) return hamming4_acc(a, b, c);
  else return sad4_acc(a, b, c);
}

__device__ __forceinline__ uint32_t imad_u32(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t d;
  asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}

// One pass of a warp over all rows of the band for 32 disparities.
// Thread tile: 8 window positions (a = 8*ul + i) x 4 disparities (j' = 4*jh + j); lane = 4*dl + ul,
// dl = 4*jh + q, q = R copy. 32 V accumulators per thread.
//
// Invalid candidates (x' outside the frame, d outside [dmin, dmax]) cost nothing extra: for a fixed
// disparity the valid windows of a phase form an interval [i0, i1) of the column index g = 8*ul + i
// (x' = xa + 4g), and a window sums the NW consecutive columns [g, g + NW). The V accumulators are
// running sums, so a constant planted at the start stays in them for the whole pass: columns
// i0-1, i0-1-NW, ... and i1+NW-1, i1+2NW-1, ... start at BIG = 2^(31-xb) instead of 0. Every invalid
// window then contains exactly one BIG column and its key carries bit 31 (true keys stay below 2^31,
// checked on the host), every valid window contains none. No per-element masks, no second code path.
template <int DIR, int NW, bool FOLD, bool RING2, int NPL, int JT, bool CENSUS, int NJ = JT>
__device__ __forceinline__ void dense_pass(const DevJob& J, const DenseCfg& cfg, uint32_t* s_ring, uint32_t* s_best,
                                           const uint32_t* __restrict__ Lg, const uint32_t* __restrict__ Rg, const int X0,
                                           const int XR0, const int run, const int dbase, const int r_shift,
                                           const int rows_in, const uint32_t minus_one) {
  // `run` is the 32-px x-run this lane works on: its own (lane & 3), or run 3 of a later pass for the guest lane
  // of a folded pass (see the kernel); `r_shift` moves the guest's R operands to that pass's disparities
  const int tid = threadIdx.x, lane = tid & 31, p = tid >> 5;
  const int ul = run, dl = lane >> 2, q = dl & 3, jh = dl >> 2;
  const int x0 = X0 + p + 32 * ul;  // window x of this thread's column i = 0 (x_i = x0 + 4i, i < 8)
  const bool guest = FOLD && (lane & 3) == 0;
  constexpr int kRB = NPL == 1 ? 4 : 2;  // rows per staging block (a ring slot holds NPL plane rows)
  constexpr int kRW = r_copy_words(JT), kRowWords = row_words(JT);
  constexpr int kSlotWords = NPL * kRowWords;
  const int th = J.th;
  const int row_words = cfg.pitch >> 2;
  const long long plane_words = cfg.plane_stride >> 2;
  const uint32_t key_scale = 1u << cfg.xb;
  const uint32_t minus_scale = key_scale * minus_one;  // -(1 << xb), kept opaque so the multiply stays an IMAD
  const uint32_t big = 1u << (31 - cfg.xb);

  // NJ = JT: the regular pass (JT disparities per thread, 8 JT per warp). NJ = 1 (JT = 4 only): the thin pass that closes a bounded range
  // (only j = 0 is computed; lanes jh = 0 carry the four disparities D0 + p - 3 .. D0 + p the regular passes of this
  // warp have not reached, lanes jh = 1 lie beyond dmax and are planted BIG) at about a third of a regular pass
  uint32_t code[NJ];
  uint32_t V[8][NJ];
#pragma unroll
  for (int j = 0; j < NJ; ++j) {
    const int d = dbase + 4 * j;
    // x' of this thread's column 0; outside [-28, nxc-1] none of its 8 windows has a valid candidate at this d:
    // the code is then parked at 0 so that it can neither wrap nor spill into the cost bits
    const int c0 = DIR < 0 ? x0 - d : x0 + d;
    code[j] = (c0 < -28 || c0 > J.nxc - 1) ? 0u : (uint32_t)(c0 + kCodeOff);
    // x' of column g = 0 of this phase; valid columns g in [i0, i1)
    const int xa = (DIR < 0 ? X0 + p - d : X0 + p + d);
    int i0 = xa >= 0 ? 0 : (-xa + 3) >> 2;
    int i1 = J.nxc - 1 - xa >= 0 ? ((J.nxc - 1 - xa) >> 2) + 1 : 0;
    if (d < J.dmin || d > J.dmax || i0 >= i1) { i0 = 1 << 20; i1 = 1 << 21; }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int g = 8 * ul + i;
      const bool is_big = (g < i0 && (i0 - 1 - g) % NW == 0) || (g >= i1 + NW - 1 && (g - (i1 + NW - 1)) % NW == 0);
      V[i][j] = is_big ? big : 0u;
    }
  }

  // ---- staging. Two ring layouts:
  //   RING2 = false (th <= 16): one ring of th + 2*kRB rows; a row is fetched once and read twice, when it enters
  //           the windows and th rows later when it leaves them.
  //   RING2 = true  (taller templates): the ring depth no longer grows with th — 2*kRB slots for the entering rows
  //           and 2*kRB for the leaving rows, each double-buffered by block of kRB rows (row r sits in slot r & 7 of
  //           its half); a row is fetched twice, th rows apart (the second fetch is an L2 hit), which leaves shared
  //           memory for tall bands (32x32 templates: 73-row bands instead of 14).
  // A block is 18 chunks of 4 words per row (8 of the L segment, 10 of the R segment), per half: thread t takes
  // task t (RING2: threads 0..15 also task 128 + t). A task turns five aligned global words into the four
  // byte-shifted copies of its chunk: 12 funnel shifts, one STS.128 per copy.
  constexpr int kChunks = kLW / 4 + r_copy_chunks(JT);
  struct StageTask {
    const uint32_t* g;  // frame rows of the band (L or R), this task's plane
    int row, back;      // row inside the block; th for the leaving half, 0 for the entering half
    int gb;             // first global word of the chunk (before clamping to the frame row)
    int off, kw;        // word offset inside the ring (half + plane + copy 0 + chunk), words between copies
    bool on;
  };
  auto make_task = [&](int k) {
    StageTask t;
    constexpr int kHalfTasks = kRB * NPL * kChunks;
    t.on = k < (RING2 ? 2 : 1) * kHalfTasks;
    const int half = k >= kHalfTasks ? 1 : 0;
    int rem = k - half * kHalfTasks;
    t.row = rem / (NPL * kChunks);
    rem -= t.row * (NPL * kChunks);
    const int pl = rem / kChunks, c = rem - pl * kChunks;
    const bool left = c < kLW / 4;
    const int w = left ? 4 * c : 4 * (c - kLW / 4);
    t.g = (left ? Lg : Rg) + (long long)pl * plane_words;
    t.back = half ? th : 0;
    t.gb = ((left ? X0 : XR0) >> 2) + w;  // X0, XR0 are multiples of 4
    t.kw = left ? kLW : kRW;
    t.off = half * 2 * kRB * kSlotWords + pl * kRowWords + (left ? 0 : 4 * kLW) + w;
    return t;
  };
  static_assert((RING2 ? 2 : 1) * kRB * NPL * kChunks <= 2 * kDenseThreads, "two staging tasks per thread");
  constexpr bool kTwoTasks = (RING2 ? 2 : 1) * kRB * NPL * kChunks > kDenseThreads;
  const StageTask task_a = make_task(tid), task_b = make_task(kDenseThreads + tid);
  const int nr = th + 2 * kRB;  // !RING2: ring depth
  int stage_slot_a = task_a.row, stage_slot_b = task_b.row;  // !RING2: ring slot of the task's row in the next block to stage
  auto run_task = [&](const StageTask& t, int row_begin, int stage_slot) {
    const int r = row_begin + t.row, gr = r - t.back;
    if (!t.on || r >= rows_in || gr < 0) return;
    const uint32_t* gp = t.g + (long long)gr * row_words;
    uint32_t w[5];
#pragma unroll
    for (int k = 0; k < 5; ++k) w[k] = __ldg(gp + min(max(t.gb + k, 0), row_words - 1));
    uint32_t* dst = s_ring + (size_t)(RING2 ? (r & (2 * kRB - 1)) : stage_slot) * kSlotWords + t.off;
    *reinterpret_cast<uint4*>(dst) = make_uint4(w[0], w[1], w[2], w[3]);
#pragma unroll
    for (int c = 1; c < 4; ++c)
      *reinterpret_cast<uint4*>(dst + c * t.kw) =
          make_uint4(__funnelshift_r(w[0], w[1], 8 * c), __funnelshift_r(w[1], w[2], 8 * c),
                     __funnelshift_r(w[2], w[3], 8 * c), __funnelshift_r(w[3], w[4], 8 * c));
  };
  auto stage = [&](int row_begin) {
    run_task(task_a, row_begin, stage_slot_a);
    if (kTwoTasks) run_task(task_b, row_begin, stage_slot_b);
    if (!RING2) {
      stage_slot_a += kRB; if (stage_slot_a >= nr) stage_slot_a -= nr;
      stage_slot_b += kRB; if (stage_slot_b >= nr) stage_slot_b -= nr;
    }
  };

  // this thread's operand words inside a ring row: L words [8ul, 8ul+8) of copy p; R words
  // [rbase, rbase+12) of copy q, element (i, j) at rbase + (DIR<0 ? i - j + 4 : i + j)
  const uint32_t* my_l = s_ring + p * kLW + 8 * ul;
  const uint32_t* my_r = s_ring + 4 * kLW + q * kRW + 8 * ul + (DIR < 0 ? JT - JT * jh : JT * jh) + r_shift;
  // the window this lane owns after the reduce-scatter min: position 8*ul + own_i
  const int own_i = ((dl >> 2) & 1) * 4 + ((dl >> 1) & 1) * 2 + (dl & 1);
  const bool b4 = (dl >> 2) & 1, b3 = (dl >> 1) & 1, b2 = dl & 1;
  uint32_t* my_best = s_best + p * 32 + 8 * ul + own_i;

  const uint32_t* my_lo = my_l + (RING2 ? 2 * kRB * kSlotWords : 0);  // RING2: the half that holds the leaving rows
  const uint32_t* my_ro = my_r + (RING2 ? 2 * kRB * kSlotWords : 0);
  int slot_new = 0, slot_old = 0;  // !RING2

  // one row of the band: the row enters the windows (V += h), the row th above leaves them (V -= h), the
  // window sums become keys and are folded into the running best. The three phases of a pass (warm-up,
  // first full window, steady state) are separate straight-line instantiations, so that the steady-state
  // body is one basic block the scheduler can interleave across the ALU and FMA pipes.
  auto row_body = [&](auto has_old_t, auto has_keys_t, int row) {
    constexpr bool HAS_OLD = decltype(has_old_t)::value, HAS_KEYS = decltype(has_keys_t)::value;
    {
      const int slot = RING2 ? (row & (2 * kRB - 1)) : slot_new;
      if (!RING2) slot_new = slot_new + 1 == nr ? 0 : slot_new + 1;
#pragma unroll
      for (int pl = 0; pl < NPL; ++pl) {
        const uint4* lp = reinterpret_cast<const uint4*>(my_l + (size_t)slot * kSlotWords + pl * kRowWords);
        const uint4* rp = reinterpret_cast<const uint4*>(my_r + (size_t)slot * kSlotWords + pl * kRowWords);
        const uint4 l0 = lp[0], l1 = lp[1];
        const uint32_t Lw[8] = {l0.x, l0.y, l0.z, l0.w, l1.x, l1.y, l1.z, l1.w};
        uint32_t Rw[JT + 8];
#pragma unroll
        for (int k = 0; k < (JT + 8) / 4; ++k) { const uint4 rr = rp[k]; Rw[4 * k] = rr.x; Rw[4 * k + 1] = rr.y; Rw[4 * k + 2] = rr.z; Rw[4 * k + 3] = rr.w; }
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < NJ; ++j) V[i][j] = cost4_acc<CENSUS>(Lw[i], Rw[DIR < 0 ? i - j + JT : i + j], V[i][j]);
      }
    }
    if (HAS_OLD) {
      const int slot = RING2 ? (row & (2 * kRB - 1)) : slot_old;
      if (!RING2) slot_old = slot_old + 1 == nr ? 0 : slot_old + 1;
      if (NPL == 1) {
        const uint4* lo = reinterpret_cast<const uint4*>(my_lo + (size_t)slot * kSlotWords);
        const uint4* ro = reinterpret_cast<const uint4*>(my_ro + (size_t)slot * kSlotWords);
        const uint4 m0 = lo[0], m1 = lo[1];
        const uint32_t Lw[8] = {m0.x, m0.y, m0.z, m0.w, m1.x, m1.y, m1.z, m1.w};
        uint32_t Rw[JT + 8];
#pragma unroll
        for (int k = 0; k < (JT + 8) / 4; ++k) { const uint4 rr = ro[k]; Rw[4 * k] = rr.x; Rw[4 * k + 1] = rr.y; Rw[4 * k + 2] = rr.z; Rw[4 * k + 3] = rr.w; }
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < NJ; ++j) {
            const uint32_t t = cost4_acc<CENSUS>(Lw[i], Rw[DIR < 0 ? i - j + JT : i + j], 0u);
            V[i][j] = imad_u32(t, minus_one, V[i][j]);  // V -= t on the FMA pipe
          }
      } else {
        uint32_t T[8][NJ <= 4 ? NJ : 1];
        // colour: with 4 disparities per thread the leaving row's |a - b| of all planes go through one temporary, so the
        // subtraction costs one IMAD per candidate slot whatever the number of planes; with 8 (64 accumulators) there are
        // no registers for the temporary and every plane subtracts on its own
#pragma unroll
        for (int pl = 0; pl < NPL; ++pl) {
          const uint4* lo = reinterpret_cast<const uint4*>(my_lo + (size_t)slot * kSlotWords + pl * kRowWords);
          const uint4* ro = reinterpret_cast<const uint4*>(my_ro + (size_t)slot * kSlotWords + pl * kRowWords);
          const uint4 m0 = lo[0], m1 = lo[1];
          const uint32_t Lw[8] = {m0.x, m0.y, m0.z, m0.w, m1.x, m1.y, m1.z, m1.w};
          uint32_t Rw[JT + 8];
#pragma unroll
          for (int k = 0; k < (JT + 8) / 4; ++k) { const uint4 rr = ro[k]; Rw[4 * k] = rr.x; Rw[4 * k + 1] = rr.y; Rw[4 * k + 2] = rr.z; Rw[4 * k + 3] = rr.w; }
          if (NJ <= 4) {
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
              for (int j = 0; j < NJ; ++j) T[i][NJ <= 4 ? j : 0] = cost4_acc<CENSUS>(Lw[i], Rw[DIR < 0 ? i - j + JT : i + j], pl == 0 ? 0u : T[i][NJ <= 4 ? j : 0]);
          } else {
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
              for (int j = 0; j < NJ; ++j) V[i][j] = imad_u32(cost4_acc<CENSUS>(Lw[i], Rw[DIR < 0 ? i - j + JT : i + j], 0u), minus_one, V[i][j]);
          }
        }
        if (NJ <= 4) {
#pragma unroll
          for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < NJ; ++j) V[i][j] = imad_u32(T[i][NJ <= 4 ? j : 0], minus_one, V[i][j]);
        }
      }
    }
    if (HAS_KEYS) {
      uint32_t best[8];
#pragma unroll
      for (int jp = 0; jp < NJ; jp += 2) {
        uint32_t key[2][8];
#pragma unroll
        for (int jj = 0; jj < (NJ == 1 ? 1 : 2); ++jj) {
          const int j = jp + jj;
          // columns 8 .. 8+NW-2 come from the next u-lane (garbage for ul = 3: those positions are not emitted)
          uint32_t Vx[8 + NW - 1];
#pragma unroll
          for (int i = 0; i < 8; ++i) Vx[i] = V[i][j];
#pragma unroll
          for (int c = 0; c < NW - 1; ++c) Vx[8 + c] = __shfl_down_sync(0xffffffffu, V[c][j], 1, 4);
          uint32_t T = Vx[0];
#pragma unroll
          for (int k = 1; k < NW; ++k) T += Vx[k];
          // slide the packed key itself: key_{i+1} = key_i + (Vx[i+NW] - Vx[i]) << xb, two IMADs on the
          // FMA pipe (wrap-around arithmetic is exact: every true key fits in 31 bits, BIG adds bit 31)
          uint32_t k = imad_u32(T, key_scale, code[j]);
          key[jj][0] = k;
#pragma unroll
          for (int i = 0; i < 7; ++i) {
            k = imad_u32(Vx[i], minus_scale, k);
            k = imad_u32(Vx[i + NW], key_scale, k);
            key[jj][i + 1] = k;
          }
        }
#pragma unroll
        for (int i = 0; i < 8; ++i)
          best[i] = NJ == 1 ? key[0][i] : jp == 0 ? min(key[0][i], key[1][i]) : __vimin3_u32(best[i], key[0][i], key[1][i]);
      }
      // reduce-scatter min over the 8 d-lanes (lane bits 4, 3, 2): 4 + 2 + 1 shuffles, each lane ends
      // with the minimum of one window
      uint32_t h4[4], h2[2], h1;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const uint32_t keep = b4 ? best[4 + k] : best[k], send = b4 ? best[k] : best[4 + k];
        h4[k] = min(keep, __shfl_xor_sync(0xffffffffu, send, 16));
      }
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        const uint32_t keep = b3 ? h4[2 + k] : h4[k], send = b3 ? h4[k] : h4[2 + k];
        h2[k] = min(keep, __shfl_xor_sync(0xffffffffu, send, 8));
      }
      {
        const uint32_t keep = b2 ? h2[1] : h2[0], send = b2 ? h2[0] : h2[1];
        h1 = min(keep, __shfl_xor_sync(0xffffffffu, send, 4));
      }
      uint32_t* bp = my_best + (size_t)(row - (th - 1)) * 128;
      if (!guest) *bp = min(*bp, h1);
      if (FOLD) {  // the guest lane shares its windows with lane 3 of the same d-lane: merge after it
        __syncwarp();
        if (guest) *bp = min(*bp, h1);
      }
    }
  };
  // every kRB rows: all warps are done with the previous block (its ring slots may be overwritten), the block
  // staged meanwhile becomes visible, and the block after it is fetched
  auto block_edge = [&](int row) {
    if ((row & (kRB - 1)) == 0) {
      __syncthreads();
      stage(row + kRB);
    }
  };

  __syncthreads();  // previous pass done with the ring; s_best init visible
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

// The body of the sweep's kernels (dense_sad_argmin_kernel, dense_census_argmin_kernel).
// DIR = -1: LeftCam (x' = x - d); DIR = +1: RightCam (x' = x + d).
// NW = tw / 4 packed words per window (2..8: the halo columns come from one neighbouring lane).
template <int DIR, int NW, bool RING2, int NPL, int JT, bool CENSUS>
__device__ __forceinline__ void dense_argmin(const DevJob& J, const DenseCfg& cfg, const uint32_t minus_one) {
  constexpr int PD = 8 * JT;  // disparities a warp covers per pass
  extern __shared__ __align__(16) uint32_t smem_u32[];
  uint32_t* s_ring = smem_u32;                                  // RING2 ? [2][2*kRB][kRowWords] : [th + 2*kRB][kRowWords]
  uint32_t* s_best = smem_u32 + cfg.ring_words;                 // [bh][4][32]

  const int tid = threadIdx.x, lane = tid & 31, p = tid >> 5;   // p: byte phase of this warp
  const int ul = lane & 3, dl = lane >> 2;
  // Block order = longest first inside chunks of pairs: a tile's work grows with the number of disparities its windows
  // can reach (LeftCam: with x, up to 20 passes against 2 for the full-range config), so inside a chunk all CTAs of the
  // heaviest tile are dispatched first and the lightest tile fills the tail (of the grid, for the last chunk). The chunk
  // (cfg.chunk_pairs, sized on the host to a fraction of L2) keeps the six tiles that read the same frame rows close in
  // time: without it every frame was fetched from DRAM once per tile (ncu: 589 MB read for 157 MB of frames).
  const int per_chunk = cfg.n_xtiles * cfg.n_bands * cfg.chunk_pairs;
  const int chunk = blockIdx.x / per_chunk, crem = blockIdx.x - chunk * per_chunk;
  const int per_tile = cfg.n_bands * min(cfg.chunk_pairs, cfg.n_pairs - chunk * cfg.chunk_pairs);
  const int t_ord = crem / per_tile, rem = crem - t_ord * per_tile;
  const int tile = DIR < 0 ? cfg.n_xtiles - 1 - t_ord : t_ord;
  const int pair = chunk * cfg.chunk_pairs + rem / cfg.n_bands, band = rem % cfg.n_bands;
  const int X0 = tile * cfg.stride_px - cfg.x_off;  // LeftCam: the partial tile sits at the low-x end (fewest disparities)
  const int y0 = band * cfg.bh;
  const int bh = min(cfg.bh, J.nyc - y0);
  const int rows_in = bh + J.th - 1;
  const uint32_t* Lg = reinterpret_cast<const uint32_t*>(cfg.lp + (long long)pair * cfg.pair_stride + (long long)y0 * cfg.pitch);
  const uint32_t* Rg = reinterpret_cast<const uint32_t*>(cfg.rp + (long long)pair * cfg.pair_stride + (long long)y0 * cfg.pitch);
  const int xb = cfg.xb;

  for (int i = tid; i < bh * 128; i += kDenseThreads) s_best[i] = 0xffffffffu;

  // disparity range this tile can use
  const int x_lo = max(X0, 0), x_hi = min(X0 + cfg.stride_px - 1, J.nxc - 1);
  int d_lo, d_hi;
  if (DIR < 0) { d_lo = max(J.dmin, x_lo - (J.nxc - 1)); d_hi = min(J.dmax, x_hi); }
  else { d_lo = max(J.dmin, -x_hi); d_hi = min(J.dmax, J.nxc - 1 - x_lo); }
  d_lo = d_lo & ~3;  // floor to a multiple of 4 (also for negatives): keeps the R copies word aligned
  // warp p, d-lane (jh, q) covers d = D0 + 16jh + 4j + (p - q) [LeftCam] / ... + (q - p) [RightCam], j < 4:
  // every warp sees 32 consecutive d starting in [D0 - 3, D0]; the shortest reach is D0 + 28.
  // Passes each 32-px x-run (x-lane) needs. LeftCam runs further right reach further (d <= x): the last passes
  // of a tile keep only runs {1,2,3}, {2,3}, {3} busy.
  int n_run[4];
  // Thin last pass: a warp's regular passes reach d_lo + 32n - 4 .. d_lo + 32n - 1 depending on its phase, so a range
  // whose length is a multiple of 32 (128, 256: the usual ones) or up to 3 short of one would need a whole extra pass
  // for its last 1 .. 3 disparities in three of the four warps. When every run of the tile is in that situation the
  // last pass is run with one disparity per thread instead of four (dense_pass<..., NJ = 1>).
  bool thin = true;
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int xl = max(X0 + 32 * r, 0), xh = min(min(X0 + 32 * r + 31, X0 + cfg.stride_px - 1), J.nxc - 1);
    int dh;
    if (DIR < 0) dh = min(J.dmax, xh); else dh = min(J.dmax, J.nxc - 1 - xl);
    n_run[r] = (xh >= xl && dh >= d_lo) ? (dh - d_lo + 3) / PD + 1 : 0;
    if (n_run[r] > 0 && dh - d_lo > PD * (n_run[r] - 1)) thin = false;  // the thin pass would not reach dh in every warp
  }
  const int n_all = max(max(n_run[0], n_run[1]), max(n_run[2], n_run[3]));
#pragma unroll
  for (int r = 0; r < 4; ++r)
    if (n_run[r] > 0 && n_run[r] != n_all) thin = false;
  if (n_all == 0) thin = false;
  // Fold (LeftCam): run 3 never uses its neighbour's columns (the tile's last 3 positions are not emitted), so
  // its lane-0 slot in a pass where run 0 is already done can host run 3 of one of the tile's last passes,
  // which then need not run at all.
  int n_fold = 0;
  // (the guest's R words sit 24 - (PD / 4) m words from its host's, m = passes between the two: m <= 3 at PD = 32, m <= 1 at PD = 64)
  if (DIR < 0 && n_run[0] <= n_run[1] && n_run[1] <= n_run[2] && n_run[2] <= n_run[3] && n_run[3] - n_run[0] <= (JT == 4 ? 3 : 2))
    n_fold = min(n_run[1] - n_run[0], n_run[3] - n_run[2]);
  const int n_pass = n_all - n_fold - (thin ? 1 : 0);  // thin implies equal runs, i.e. no fold

  for (int pass = 0; pass < n_pass; ++pass) {
    const int D0 = d_lo + PD * pass;
    const bool fold_pass = pass >= n_run[0] && pass < n_run[0] + n_fold;
    const bool guest = fold_pass && ul == 0;
    const int run = guest ? 3 : ul;
    const int D0_mine = guest ? d_lo + PD * (n_all - 1 - (pass - n_run[0])) : D0;
    // d of (this lane, j = 0); d_j = dbase + 4j, j < 4. dl = 4*jh + q: R copy q, upper/lower half of the 8 d-steps
    const int dbase = D0_mine + 4 * JT * (dl >> 2) + (DIR < 0 ? (p - (dl & 3)) : ((dl & 3) - p));
    // first byte of the R copies for this pass: R copy q word w = bytes [XR0 + q + 4w, +4)
    const int XR0 = DIR < 0 ? X0 - D0 - PD : X0 + D0;
    const int r_shift = DIR < 0 ? -((D0_mine - D0) >> 2) : ((D0_mine - D0) >> 2);
    if (fold_pass) dense_pass<DIR, NW, true, RING2, NPL, JT, CENSUS>(J, cfg, s_ring, s_best, Lg, Rg, X0, XR0, run, dbase, r_shift, rows_in, minus_one);
    else dense_pass<DIR, NW, false, RING2, NPL, JT, CENSUS>(J, cfg, s_ring, s_best, Lg, Rg, X0, XR0, run, dbase, r_shift, rows_in, minus_one);
  }
  if (thin) {
    const int D0 = d_lo + PD * n_pass;
    const int dbase = D0 + 4 * JT * (dl >> 2) + (DIR < 0 ? (p - (dl & 3)) : ((dl & 3) - p));
    const int XR0 = DIR < 0 ? X0 - D0 - PD : X0 + D0;
    dense_pass<DIR, NW, false, RING2, NPL, JT, CENSUS, 1>(J, cfg, s_ring, s_best, Lg, Rg, X0, XR0, ul, dbase, 0, rows_in, minus_one);
  }
  __syncthreads();

  // ---- fused epilogue: key -> (cost, x') -> Match / disparity / distance
  const int n_pos = 32 - NW + 1;  // valid window positions per phase in a tile
  const int span = min(cfg.stride_px, J.nxc - X0);
  const uint32_t code_mask = (1u << xb) - 1;
  for (int idx = tid; idx < bh * span; idx += kDenseThreads) {
    const int yy = idx / span, xo = idx - yy * span;
    const int pp = xo & 3, a = xo >> 2;
    if (a >= n_pos || X0 + xo < 0) continue;
    const uint32_t key = s_best[((size_t)yy * 4 + pp) * 32 + a];
    const int x = X0 + xo, y = y0 + yy;
    const long long w = (long long)y * J.nx + x;
    const long long g = (long long)(cfg.pair0 + pair) * J.n_templates + w;
    if (key & 0x80000000u) {  // untouched (~0) or only invalid candidates
      write_result(J, g, (uint32_t)w, x, y, -1, 0xffffffffu, 0.0, __longlong_as_double(0x7ff0000000000000ll));
    } else {
      const uint32_t raw = key >> xb;
      const int c = (int)(key & code_mask) - kCodeOff;  // = x0 -/+ d of the owning thread column 0
      const int xr = c + 4 * (a & 7);
      write_result(J, g, (uint32_t)w, x, y, xr, raw, 0.0, normalised_cost(raw, CENSUS ? USV_COST_CENSUS : USV_COST_SAD, J.n_elems));
    }
  }
}

template <int DIR, int NW, bool RING2, int NPL, int JT>
__global__ void __launch_bounds__(kDenseThreads, NPL == 1 && JT == 4 ? 4 : 3)
dense_sad_argmin_kernel(const DevJob J, const DenseCfg cfg, const uint32_t minus_one) {
  dense_argmin<DIR, NW, RING2, NPL, JT, false>(J, cfg, minus_one);
}
template <int DIR, int NW, bool RING2, int NPL, int JT>
__global__ void __launch_bounds__(kDenseThreads, NPL == 1 && JT == 4 ? 4 : 3)
dense_census_argmin_kernel(const DevJob J, const DenseCfg cfg, const uint32_t minus_one) {
  dense_argmin<DIR, NW, RING2, NPL, JT, true>(J, cfg, minus_one);
}

// The kernel of the <NPL, JT, CENSUS> variant for one direction, template width and ring kind (colour frames always run
// the two-half ring). dense_kernel is explicitly instantiated once per variant, in the translation unit that compiles it.
using DenseKernel = void (*)(DevJob, DenseCfg, uint32_t);
template <int DIR, int NW, bool RING2, int NPL, int JT, bool CENSUS>
DenseKernel dense_kernel_cost() {
  if constexpr (CENSUS) return dense_census_argmin_kernel<DIR, NW, RING2, NPL, JT>;
  else return dense_sad_argmin_kernel<DIR, NW, RING2, NPL, JT>;
}
template <int DIR, int NW, int NPL, int JT, bool CENSUS>
DenseKernel dense_kernel_ring(bool ring2) {
  if constexpr (NPL > 1) return dense_kernel_cost<DIR, NW, true, NPL, JT, CENSUS>();
  else return ring2 ? dense_kernel_cost<DIR, NW, true, NPL, JT, CENSUS>() : dense_kernel_cost<DIR, NW, false, NPL, JT, CENSUS>();
}
template <int DIR, int NPL, int JT, bool CENSUS>
DenseKernel dense_kernel_nw(int nw, bool ring2) {
  switch (nw) {
    case 2: return dense_kernel_ring<DIR, 2, NPL, JT, CENSUS>(ring2);
    case 3: return dense_kernel_ring<DIR, 3, NPL, JT, CENSUS>(ring2);
    case 4: return dense_kernel_ring<DIR, 4, NPL, JT, CENSUS>(ring2);
    case 6: return dense_kernel_ring<DIR, 6, NPL, JT, CENSUS>(ring2);
    default: return dense_kernel_ring<DIR, 8, NPL, JT, CENSUS>(ring2);
  }
}
template <int NPL, int JT, bool CENSUS = false>
DenseKernel dense_kernel(int dir, int nw, bool ring2) {
  return dir < 0 ? dense_kernel_nw<-1, NPL, JT, CENSUS>(nw, ring2) : dense_kernel_nw<1, NPL, JT, CENSUS>(nw, ring2);
}

}  // namespace usv
