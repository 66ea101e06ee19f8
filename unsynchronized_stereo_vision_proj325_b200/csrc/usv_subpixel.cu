// usv_subpixel.cu — sub-pixel refinement of dense-sweep winners (include/usv_b200.h, usv_refine_subpixel_device).
//
// One thread per window of the dense grid, consecutive threads on consecutive windows of one row; one CTA per (strip of
// 128 windows, row, pair). The thread reads the winner's RightIndex x*, recomputes the three candidates x*-1, x*, x*+1
// in direct form, and fits the parabola through their costs (DESIGN §4.8). The three candidate byte streams are the
// same right-frame row shifted by 0, C and 2C bytes, so one aligned word load per template word feeds all three: the
// word at the candidate x*-1 comes from one funnel shift, the other two from one more shift of that stream (or none).
//   SAD : VABSDIFF4 (sad4_acc)            SSD : VABSDIFF4 + IDP.4A
//   NCC / ZNCC: IDP.4A for Sab, Sb, Sbb of each candidate, Sa / Saa of the template once
// Frames are read straight from global memory through L1: neighbouring windows share almost all their words. Only words
// that hold a byte of [0, width*C) are loaded, and bytes past the template row are masked, so row padding never reaches
// a cost.
#include "usv_common.cuh"

namespace usv {

constexpr int kSubpixelThreads = 128;

struct SubpixelJob {
  const uint8_t* left;
  const uint8_t* right;
  long long frame_stride;
  int row_stride, tw, th, dmin, dmax, sx, sy, nx, ny, nxc, camera_side, distance_kind, n_elems;
  const uint32_t* right_index;
  int* disparity_x16;
  double* distance;
};

// words of the candidates x*-1, x*, x*+1 (byte offsets 0, C, 2C) from three consecutive words of the x*-1 stream
template <int C>
__device__ __forceinline__ void cand_words(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t& b0, uint32_t& b1, uint32_t& b2) {
  b0 = c0;
  if (C == 1) { b1 = __funnelshift_r(c0, c1, 8); b2 = __funnelshift_r(c0, c1, 16); }
  else if (C == 2) { b1 = __funnelshift_r(c0, c1, 16); b2 = c1; }
  else if (C == 3) { b1 = __funnelshift_r(c0, c1, 24); b2 = __funnelshift_r(c1, c2, 16); }
  else { b1 = c1; b2 = c2; }
}

struct Acc3 {
  uint32_t c[3];   // SAD / SSD cost, or Sab (NCC / ZNCC)
  uint32_t sb[3], sbb[3];
  uint32_t sa, saa;
};

template <int KIND>
__device__ __forceinline__ void acc_word(Acc3& A, uint32_t a, uint32_t b0, uint32_t b1, uint32_t b2) {
  const uint32_t b[3] = {b0, b1, b2};
  if (KIND >= USV_COST_NCC) {
    A.sa = __dp4a(a, 0x01010101u, A.sa);
    A.saa = __dp4a(a, a, A.saa);
  }
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    if (KIND == USV_COST_SAD) {
      A.c[j] = sad4_acc(a, b[j], A.c[j]);
    } else if (KIND == USV_COST_SSD) {
      const uint32_t d = __vabsdiffu4(a, b[j]);
      A.c[j] = __dp4a(d, d, A.c[j]);
    } else {
      A.c[j] = __dp4a(a, b[j], A.c[j]);
      A.sb[j] = __dp4a(b[j], 0x01010101u, A.sb[j]);
      A.sbb[j] = __dp4a(b[j], b[j], A.sbb[j]);
    }
  }
}

template <int KIND, int C>
__global__ void __launch_bounds__(kSubpixelThreads) subpixel_refine_kernel(const SubpixelJob J) {
  const int ix = blockIdx.x * kSubpixelThreads + threadIdx.x;
  if (ix >= J.nx) return;
  const int pair = blockIdx.z;
  const int rb = J.tw * C;                  // template bytes per row
  const int nw = (rb + 3) >> 2;             // template words per row
  const uint32_t tail = (rb & 3) ? (0xffffffffu >> (32 - 8 * (rb & 3))) : 0xffffffffu;
  for (int iy = blockIdx.y; iy < J.ny; iy += gridDim.y) {
    const int x = ix * J.sx, y = iy * J.sy;
    const long long g = ((long long)pair * J.ny + iy) * J.nx + ix;
    const uint32_t r = J.right_index[g];
    int x16 = USV_NO_SUBPIXEL;
    double dist = 0.0;
    int lo, hi;
    cand_range(x, J.nxc, J.camera_side, J.dmin, J.dmax, &lo, &hi);
    const int xs = (int)(r % (uint32_t)J.nxc);
    // a refinement target is a candidate of this window: same row, x* inside the window's clipped range
    if (r != USV_NO_MATCH && r / (uint32_t)J.nxc == (uint32_t)y && xs >= lo && xs <= hi) {
      const int d = J.camera_side == USV_LEFT_CAM ? x - xs : xs - x;
      int q = 0;
      if (xs - 1 >= lo && xs + 1 <= hi) {
        const uint8_t* Lf = J.left + (long long)pair * J.frame_stride;
        const uint8_t* Rf = J.right + (long long)pair * J.frame_stride;
        const int bl = x * C, br = (xs - 1) * C;
        const int lw = bl >> 2, lsh = (bl & 3) * 8, llast = (bl + rb - 1) >> 2;
        const int rw = br >> 2, rsh = (br & 3) * 8, rlast = (br + 2 * C + rb - 1) >> 2;
        Acc3 A;
#pragma unroll
        for (int j = 0; j < 3; ++j) A.c[j] = A.sb[j] = A.sbb[j] = 0;
        A.sa = A.saa = 0;
        for (int row = 0; row < J.th; ++row) {
          const uint32_t* Lp = reinterpret_cast<const uint32_t*>(Lf + (long long)(y + row) * J.row_stride);
          const uint32_t* Rp = reinterpret_cast<const uint32_t*>(Rf + (long long)(y + row) * J.row_stride);
          uint32_t l0 = __ldg(Lp + lw), l1 = __ldg(Lp + min(lw + 1, llast));
          const uint32_t q0 = __ldg(Rp + rw), q1 = __ldg(Rp + min(rw + 1, rlast)), q2 = __ldg(Rp + min(rw + 2, rlast));
          uint32_t qn = __ldg(Rp + min(rw + 3, rlast));
          uint32_t c0 = __funnelshift_r(q0, q1, rsh), c1 = __funnelshift_r(q1, q2, rsh), c2 = __funnelshift_r(q2, qn, rsh);
          for (int k = 0; k < nw - 1; ++k) {
            uint32_t b0, b1, b2;
            cand_words<C>(c0, c1, c2, b0, b1, b2);
            acc_word<KIND>(A, __funnelshift_r(l0, l1, lsh), b0, b1, b2);
            l0 = l1; l1 = __ldg(Lp + min(lw + k + 2, llast));
            const uint32_t qm = __ldg(Rp + min(rw + k + 4, rlast));
            c0 = c1; c1 = c2; c2 = __funnelshift_r(qn, qm, rsh); qn = qm;
          }
          uint32_t b0, b1, b2;
          cand_words<C>(c0, c1, c2, b0, b1, b2);
          acc_word<KIND>(A, __funnelshift_r(l0, l1, lsh) & tail, b0 & tail, b1 & tail, b2 & tail);
        }
        if (KIND <= USV_COST_SSD) {
          const long long cm = A.c[0], c0 = A.c[1], cp = A.c[2];
          const long long num = cm - cp, den = cm + cp - 2 * c0;
          if (den > 0) {
            const long long an = num < 0 ? -num : num;
            long long m = (16 * an + den) / (2 * den);
            if (m > 8) m = 8;
            q = (int)(num < 0 ? -m : m);
          }
        } else {
          double v[3];
#pragma unroll
          for (int j = 0; j < 3; ++j) {
            const double sc = KIND == USV_COST_NCC
                                  ? ncc_score((long long)A.c[j], (long long)A.saa, (long long)A.sbb[j])
                                  : zncc_score(J.n_elems, (long long)A.c[j], (long long)A.sa, (long long)A.sb[j],
                                               (long long)A.saa, (long long)A.sbb[j]);
            v[j] = __dsub_rn(1.0, sc);
          }
          const double num = __dsub_rn(v[0], v[2]);
          const double den = __dadd_rn(__dsub_rn(v[0], v[1]), __dsub_rn(v[2], v[1]));
          if (den > 0.0) {
            double t = round(__ddiv_rn(__dmul_rn(8.0, num), den));
            t = t > 8.0 ? 8.0 : (t < -8.0 ? -8.0 : t);
            q = (int)t;
          }
        }
      }
      x16 = J.camera_side == USV_LEFT_CAM ? 16 * d - q : 16 * d + q;
      dist = distance_from_disparity(__ddiv_rn((double)x16, 16.0), J.distance_kind);
    }
    if (J.disparity_x16) J.disparity_x16[g] = x16;
    if (J.distance) J.distance[g] = dist;
  }
}

template <int KIND>
static cudaError_t launch_subpixel_k(const SubpixelJob& J, int channels, dim3 grid, cudaStream_t st) {
  switch (channels) {
    case 1: subpixel_refine_kernel<KIND, 1><<<grid, kSubpixelThreads, 0, st>>>(J); break;
    case 2: subpixel_refine_kernel<KIND, 2><<<grid, kSubpixelThreads, 0, st>>>(J); break;
    case 3: subpixel_refine_kernel<KIND, 3><<<grid, kSubpixelThreads, 0, st>>>(J); break;
    case 4: subpixel_refine_kernel<KIND, 4><<<grid, kSubpixelThreads, 0, st>>>(J); break;
    default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

cudaError_t launch_subpixel_refine(const DevJob& D, int n_pairs, const uint32_t* d_right_index, int* d_x16, double* d_dist,
                                   cudaStream_t st) {
  SubpixelJob J;
  J.left = D.left; J.right = D.right; J.frame_stride = D.frame_stride;
  J.row_stride = D.row_stride; J.tw = D.tw; J.th = D.th; J.dmin = D.dmin; J.dmax = D.dmax; J.sx = D.sx; J.sy = D.sy;
  J.nx = D.nx; J.ny = D.ny; J.nxc = D.nxc; J.camera_side = D.camera_side; J.distance_kind = D.distance_kind;
  J.n_elems = D.n_elems;
  J.right_index = d_right_index; J.disparity_x16 = d_x16; J.distance = d_dist;
  const dim3 grid((unsigned)((D.nx + kSubpixelThreads - 1) / kSubpixelThreads), (unsigned)(D.ny < 65535 ? D.ny : 65535),
                  (unsigned)n_pairs);
  switch (D.cost_kind) {
    case USV_COST_SAD: return launch_subpixel_k<USV_COST_SAD>(J, D.channels, grid, st);
    case USV_COST_SSD: return launch_subpixel_k<USV_COST_SSD>(J, D.channels, grid, st);
    case USV_COST_NCC: return launch_subpixel_k<USV_COST_NCC>(J, D.channels, grid, st);
    case USV_COST_ZNCC: return launch_subpixel_k<USV_COST_ZNCC>(J, D.channels, grid, st);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace usv
