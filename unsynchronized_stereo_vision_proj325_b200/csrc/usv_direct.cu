// usv_direct.cu — direct-form block search for sm_100a.
//
// One CTA per (template, frame pair). The template and the search strip are
// staged in shared memory with cp.async (16-byte LDGSTS); every thread scores
// four candidates x', x'+4, x'+8, x'+12 (same byte phase, so one funnel shift
// aligns the strip words for all four) with packed-byte intrinsics:
//   SAD : __vsadu4            -> VABSDIFF4.U8.ACC
//   SSD : __vabsdiffu4+__dp4a -> VABSDIFF4.U8 + IDP.4A.U8.U8
//   NCC / ZNCC: three __dp4a  -> exact integer sum(ab), sum(b), sum(b^2)
//   CENSUS: __popc(a ^ b)     -> LOP3 + POPC, over census frames (usv_census.cu) transformed into the pair scratch
// Selection is a warp-shuffle + block argmin on a packed (cost, scan index) key,
// so "smallest cost, then earliest candidate" (P/Main.cpp:451) is one unsigned
// min and cannot depend on reduction order. The epilogue turns the winner into a
// Match record, disparity and distance (P/Main.cpp:681-694, P/DistanceCalculator.cpp:84).
//
// This is the general path (sparse template lists, any stride / template size /
// channel count, optional dump of every candidate's cost). Dense stride-1 jobs that a
// sliding-window sweep covers go to that sweep instead (DESIGN §4, usv_capi.cu: plan_match).
#include <algorithm>

#include "usv_common.cuh"

namespace usv {

constexpr int kDirectThreads = 128;
constexpr int kCandPerThread = 4;
constexpr int kChunkCands = kDirectThreads * kCandPerThread;  // candidates per CTA pass
constexpr int kStripBudget = 64 * 1024;                        // bytes of smem for strip rows

struct BestInt { unsigned long long key; };

__device__ __forceinline__ unsigned long long warp_min_u64(unsigned long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    unsigned long long t = __shfl_xor_sync(0xffffffffu, v, o);
    v = t < v ? t : v;
  }
  return v;
}

// lexicographic (value, index) min for the f64 costs
__device__ __forceinline__ void warp_min_f64(double& v, unsigned& j, long long& aux0, long long& aux1) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    double tv = __shfl_xor_sync(0xffffffffu, v, o);
    unsigned tj = __shfl_xor_sync(0xffffffffu, j, o);
    long long t0 = __shfl_xor_sync(0xffffffffu, aux0, o);
    long long t1 = __shfl_xor_sync(0xffffffffu, aux1, o);
    if (tv < v || (tv == v && tj < j)) { v = tv; j = tj; aux0 = t0; aux1 = t1; }
  }
}

template <int KIND, int C>
__global__ void __launch_bounds__(kDirectThreads)
block_cost_argmin_direct(const DevJob J, int tmpl_pitch_words, int strip_pitch_words, int rows_per_chunk) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint32_t* s_tmpl = reinterpret_cast<uint32_t*>(smem_raw);                 // [th][tmpl_pitch_words]
  uint32_t* s_strip = s_tmpl + (((size_t)J.th * tmpl_pitch_words + 3) & ~(size_t)3);  // [rows_per_chunk][strip_pitch_words], 16-B aligned
  __shared__ unsigned long long s_red[kDirectThreads / 32];
  __shared__ double s_redv[kDirectThreads / 32];
  __shared__ unsigned s_redj[kDirectThreads / 32];
  __shared__ long long s_reda[kDirectThreads / 32][2];
  __shared__ long long s_tsum[2];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int t_idx = blockIdx.x, pair = blockIdx.y;
  int x, y;
  if (J.tx) { x = J.tx[t_idx]; y = J.ty[t_idx]; }
  else { x = (t_idx % J.nx) * J.sx; y = (t_idx / J.nx) * J.sy; }
  const long long g = (long long)pair * J.n_templates + t_idx;
  // the device-pointer API cannot validate a template list that lives in HBM: a template that does not fit the frame
  // gets the "no candidate" record (USV_NO_MATCH, MatchValue +inf) instead of an out-of-bounds strip (block-uniform exit)
  if (x < 0 || x >= J.nxc || y < 0 || y >= J.nyc) {
    if (tid == 0) write_result(J, g, (uint32_t)t_idx, x, y, -1, 0xffffffffu, 0.0, __longlong_as_double(0x7ff0000000000000ll));
    return;
  }
  const uint8_t* L = J.left + (long long)pair * J.frame_stride;
  const uint8_t* R = J.right + (long long)pair * J.frame_stride;

  int lo, hi;
  cand_range(x, J.nxc, J.camera_side, J.dmin, J.dmax, &lo, &hi);
  const int nw = (J.row_bytes + 3) >> 2;  // template words per row
  const uint32_t tail_mask = (J.row_bytes & 3) ? (0xffffffffu >> (32 - 8 * (J.row_bytes & 3))) : 0xffffffffu;

  // ---- stage the template (whole, once): 16-byte cp.async from the aligned rows
  {
    const int b0 = x * C;                    // first template byte in the row
    const int a0 = b0 & ~15;                 // aligned start
    const int nchunk = ((b0 + J.row_bytes + 15) >> 4) - (a0 >> 4);
    // staged at s_strip temporarily (aligned copy), then realigned into s_tmpl
    unsigned char* tmp = reinterpret_cast<unsigned char*>(s_strip);
    const int tmp_pitch = nchunk * 16;
    for (int i = tid; i < J.th * nchunk; i += kDirectThreads) {
      int r = i / nchunk, c = i - r * nchunk;
      cp_async16(tmp + r * tmp_pitch + c * 16, L + (long long)(y + r) * J.row_stride + a0 + c * 16);
    }
    cp_async_commit();
    cp_async_wait_all();
    __syncthreads();
    const int sh = b0 - a0;
    for (int i = tid; i < J.th * nw; i += kDirectThreads) {
      int r = i / nw, k = i - r * nw;
      const unsigned char* p = tmp + r * tmp_pitch + sh + 4 * k;
      uint32_t w = 0;
      int nbytes = min(4, J.row_bytes - 4 * k);
      for (int b = 0; b < nbytes; ++b) w |= (uint32_t)p[b] << (8 * b);
      s_tmpl[r * tmpl_pitch_words + k] = w;  // zero-padded tail => masked bytes contribute 0
    }
    __syncthreads();
  }

  // integer costs (SAD, SSD, census) select on a packed (cost, index) key, correlation costs on an f64 value
  constexpr bool kInteger = KIND == USV_COST_SAD || KIND == USV_COST_SSD || KIND == USV_COST_CENSUS;

  // ---- template sums (NCC / ZNCC only)
  long long t_sa = 0, t_saa = 0;
  if (!kInteger) {
    unsigned a1 = 0, a2 = 0;
    for (int i = tid; i < J.th * nw; i += kDirectThreads) {
      int r = i / nw, k = i - r * nw;
      uint32_t w = s_tmpl[r * tmpl_pitch_words + k];
      a1 = __dp4a(w, 0x01010101u, a1);
      a2 = __dp4a(w, w, a2);
    }
    unsigned long long pk1 = a1, pk2 = a2;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      pk1 += __shfl_xor_sync(0xffffffffu, pk1, o);
      pk2 += __shfl_xor_sync(0xffffffffu, pk2, o);
    }
    if (lane == 0) { s_reda[warp][0] = (long long)pk1; s_reda[warp][1] = (long long)pk2; }
    __syncthreads();
    if (tid == 0) {
      long long u = 0, v = 0;
      for (int w = 0; w < kDirectThreads / 32; ++w) { u += s_reda[w][0]; v += s_reda[w][1]; }
      s_tsum[0] = u; s_tsum[1] = v;
    }
    __syncthreads();
    t_sa = s_tsum[0]; t_saa = s_tsum[1];
    __syncthreads();
  }

  // per-thread running best
  unsigned long long best_key = ~0ull;         // integer kinds: (cost << 32) | j
  double best_v = __longlong_as_double(0x7ff0000000000000ll);  // +inf; float kinds
  unsigned best_j = 0xffffffffu;
  long long best_a0 = 0, best_a1 = 0;          // (score bits) carried along

  const int ncand = hi >= lo ? hi - lo + 1 : 0;
  for (int c0 = 0; c0 < ncand; c0 += kChunkCands) {
    const int c1 = min(ncand, c0 + kChunkCands);           // candidates [c0, c1) of this pass
    const int xs0 = lo + c0;                                // first candidate x'
    const int sb0 = (xs0 * C) & ~15;                        // aligned strip start byte
    const int sb1 = (((lo + c1 - 1 + J.tw) * C) + 15) & ~15;
    const int nchunk16 = (sb1 - sb0) >> 4;

    // candidates of this thread: j = c0 + 16*(tid>>2) + (tid&3) + 4*i
    const int jb = c0 + 16 * (tid >> 2) + (tid & 3);
    uint32_t acc[kCandPerThread], accb[kCandPerThread], accbb[kCandPerThread];
    int woff[kCandPerThread];
    int shift_bits;
    {
      // clamp out-of-range candidates onto the last valid one (result discarded)
      int xc0 = min(lo + jb, hi);
      int boff = xc0 * C - sb0;
      shift_bits = (boff & 3) * 8;
#pragma unroll
      for (int i = 0; i < kCandPerThread; ++i) {
        int xc = min(lo + jb + 4 * i, hi);
        woff[i] = (xc * C - sb0) >> 2;  // same byte phase for every i (4*C is a multiple of 4)
        acc[i] = accb[i] = accbb[i] = 0;
      }
    }

    for (int r0 = 0; r0 < J.th; r0 += rows_per_chunk) {
      const int nr = min(rows_per_chunk, J.th - r0);
      __syncthreads();  // previous chunk fully consumed
      for (int i = tid; i < nr * nchunk16; i += kDirectThreads) {
        int r = i / nchunk16, c = i - r * nchunk16;
        cp_async16(reinterpret_cast<unsigned char*>(s_strip + (size_t)r * strip_pitch_words) + c * 16,
                   R + (long long)(y + r0 + r) * J.row_stride + sb0 + c * 16);
      }
      cp_async_commit();
      cp_async_wait_all();
      __syncthreads();

      for (int r = 0; r < nr; ++r) {
        const uint32_t* trow = s_tmpl + (size_t)(r0 + r) * tmpl_pitch_words;
        const uint32_t* srow = s_strip + (size_t)r * strip_pitch_words;
#pragma unroll 4
        for (int k = 0; k < nw; ++k) {
          const uint32_t a = trow[k];
          const uint32_t m = (k == nw - 1) ? tail_mask : 0xffffffffu;
#pragma unroll
          for (int i = 0; i < kCandPerThread; ++i) {
            uint32_t w0 = srow[woff[i] + k], w1 = srow[woff[i] + k + 1];
            uint32_t b = __funnelshift_r(w0, w1, shift_bits) & m;
            if (KIND == USV_COST_SAD) {
              acc[i] = sad4_acc(a, b, acc[i]);
            } else if (KIND == USV_COST_SSD) {
              uint32_t d = __vabsdiffu4(a, b);
              acc[i] = __dp4a(d, d, acc[i]);
            } else if (KIND == USV_COST_CENSUS) {
              acc[i] = hamming4_acc(a, b, acc[i]);
            } else {
              acc[i] = __dp4a(a, b, acc[i]);
              accb[i] = __dp4a(b, 0x01010101u, accb[i]);
              accbb[i] = __dp4a(b, b, accbb[i]);
            }
          }
        }
      }
    }

    // ---- fold this pass into the running best, optionally dump every cost
#pragma unroll
    for (int i = 0; i < kCandPerThread; ++i) {
      const int j = jb + 4 * i;
      if (j >= c1) continue;
      if (kInteger) {
        unsigned long long key = ((unsigned long long)acc[i] << 32) | (unsigned)j;
        best_key = key < best_key ? key : best_key;
        if (J.cost_rows && j < J.row_cap) J.cost_rows[g * J.row_cap + j] = acc[i];
      } else {
        double sc = KIND == USV_COST_NCC
                        ? ncc_score((long long)acc[i], t_saa, (long long)accbb[i])
                        : zncc_score(J.n_elems, (long long)acc[i], t_sa, (long long)accb[i], t_saa, (long long)accbb[i]);
        double v = __dsub_rn(1.0, sc);
        if (v < best_v || (v == best_v && (unsigned)j < best_j)) {
          best_v = v; best_j = (unsigned)j; best_a0 = __double_as_longlong(sc); best_a1 = 0;
        }
        if (J.score_rows && j < J.row_cap) J.score_rows[g * J.row_cap + j] = sc;
      }
    }
  }

  // ---- block argmin (deterministic: pure min on the packed key)
  if (kInteger) {
    unsigned long long k = warp_min_u64(best_key);
    if (lane == 0) s_red[warp] = k;
    __syncthreads();
    if (tid == 0) {
      for (int w = 1; w < kDirectThreads / 32; ++w) k = s_red[w] < k ? s_red[w] : k;
      const bool has = ncand > 0;
      const uint32_t raw = has ? (uint32_t)(k >> 32) : 0xffffffffu;
      const int bx = has ? lo + (int)(k & 0xffffffffu) : -1;
      const double value = has ? normalised_cost(raw, KIND, J.n_elems) : __longlong_as_double(0x7ff0000000000000ll);
      write_result(J, g, (uint32_t)t_idx, x, y, bx, raw, 0.0, value);
    }
  } else {
    warp_min_f64(best_v, best_j, best_a0, best_a1);
    if (lane == 0) { s_redv[warp] = best_v; s_redj[warp] = best_j; s_reda[warp][0] = best_a0; }
    __syncthreads();
    if (tid == 0) {
      double v = s_redv[0]; unsigned j = s_redj[0]; long long a0 = s_reda[0][0];
      for (int w = 1; w < kDirectThreads / 32; ++w) {
        if (s_redv[w] < v || (s_redv[w] == v && s_redj[w] < j)) { v = s_redv[w]; j = s_redj[w]; a0 = s_reda[w][0]; }
      }
      const bool has = ncand > 0 && j != 0xffffffffu;
      write_result(J, g, (uint32_t)t_idx, x, y, has ? lo + (int)j : -1, 0xffffffffu,
                   has ? __longlong_as_double(a0) : 0.0, v);
    }
  }
}

// ---- host-side launcher ----------------------------------------------------
struct DirectLayout {
  int tmpl_pitch_words, strip_pitch_words, rows;
  size_t smem;  // 0: the job does not fit the shared memory of one CTA
};

static DirectLayout direct_layout(const DevJob& J) {
  DirectLayout d;
  const int nw = (J.row_bytes + 3) / 4;
  // odd pitch in words avoids bank conflicts; the whole template area is padded to 16 B so the
  // strip area that follows it stays cp.async (16-byte) aligned
  d.tmpl_pitch_words = nw + 1;
  // widest strip a pass can need: (chunk candidates + template) bytes + alignment slack
  int max_c = J.nxc < kChunkCands ? J.nxc : kChunkCands;
  int strip_bytes = ((max_c + J.tw) * J.channels + 47) & ~15;
  d.strip_pitch_words = strip_bytes / 4 + 4;  // +16 B slack: the funnel shift reads one word ahead
  // the template's aligned staging copy temporarily lives in the strip area
  size_t tmpl_stage_bytes = (size_t)J.th * (((J.row_bytes + 15 + 16) & ~15) + 16);
  d.rows = kStripBudget / (d.strip_pitch_words * 4);
  d.smem = 0;
  if (d.rows < 1) return d;
  if (d.rows > J.th) d.rows = J.th;
  size_t strip_area = (size_t)d.rows * d.strip_pitch_words * 4;
  if (strip_area < tmpl_stage_bytes) strip_area = tmpl_stage_bytes;
  size_t smem = ((((size_t)J.th * d.tmpl_pitch_words + 3) & ~(size_t)3) * 4) + strip_area;
  smem = (smem + 15) & ~(size_t)15;
  if (smem <= 200 * 1024) d.smem = smem;
  return d;
}

// the whole template and one strip chunk must fit one CTA's shared memory (narrow, tall templates may not)
bool direct_supported(const DevJob& J) { return direct_layout(J).smem != 0; }

template <int KIND>
static cudaError_t launch_direct_c(const DevJob& J, int n_pairs, cudaStream_t st) {
  const DirectLayout d = direct_layout(J);
  if (d.smem == 0 || J.channels < 1 || J.channels > 4) return cudaErrorInvalidValue;
  const auto k = J.channels == 1 ? block_cost_argmin_direct<KIND, 1>
               : J.channels == 2 ? block_cost_argmin_direct<KIND, 2>
               : J.channels == 3 ? block_cost_argmin_direct<KIND, 3>
                                 : block_cost_argmin_direct<KIND, 4>;
  return launch_kernel(k, dim3(J.n_templates, n_pairs), dim3(kDirectThreads), d.smem, st, J, d.tmpl_pitch_words, d.strip_pitch_words, d.rows);
}

// census: the pairs run in chunks of what the scratch holds (at least one pair's census frames, usv_common.cuh:
// census_scratch_bytes_per_pair); each chunk is transformed, then scored with its outputs offset to its first pair
static cudaError_t launch_direct_census(const DevJob& J, int n_pairs, void* d_scratch, size_t scratch_bytes, cudaStream_t st,
                                        int* n_launches) {
  const int chunk = (int)std::min<size_t>((size_t)n_pairs, scratch_bytes / census_scratch_bytes_per_pair(J));
  if (chunk < 1) return cudaErrorInvalidValue;
  for (int p0 = 0; p0 < n_pairs; p0 += chunk) {
    const int np = std::min(chunk, n_pairs - p0);
    DevJob Jc;
    cudaError_t e = census_chunk(J, p0, np, (uint8_t*)d_scratch, st, Jc, n_launches);
    if (e != cudaSuccess) return e;
    const long long off = (long long)p0 * J.n_templates;
    usv_outputs& o = Jc.out;
    if (o.matches) o.matches += off;
    if (o.right_index) o.right_index += off;
    if (o.raw_cost) o.raw_cost += off;
    if (o.raw_cost_u16) o.raw_cost_u16 += off;
    if (o.score) o.score += off;
    if (o.distance) o.distance += off;
    if (o.distance_f32) o.distance_f32 += off;
    if (o.disparity_u16) o.disparity_u16 += off;
    if (Jc.cost_rows) Jc.cost_rows += off * Jc.row_cap;
    if (Jc.score_rows) Jc.score_rows += off * Jc.row_cap;
    if ((e = launch_direct_c<USV_COST_CENSUS>(Jc, np, st)) != cudaSuccess) return e;
    *n_launches += 1;
  }
  return cudaSuccess;
}

cudaError_t launch_direct(const DevJob& J, int n_pairs, void* d_scratch, size_t scratch_bytes, cudaStream_t st, int* n_launches) {
  if (J.cost_kind == USV_COST_CENSUS) return launch_direct_census(J, n_pairs, d_scratch, scratch_bytes, st, n_launches);
  *n_launches += 1;
  switch (J.cost_kind) {
    case USV_COST_SAD: return launch_direct_c<USV_COST_SAD>(J, n_pairs, st);
    case USV_COST_SSD: return launch_direct_c<USV_COST_SSD>(J, n_pairs, st);
    case USV_COST_NCC: return launch_direct_c<USV_COST_NCC>(J, n_pairs, st);
    case USV_COST_ZNCC: return launch_direct_c<USV_COST_ZNCC>(J, n_pairs, st);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace usv
