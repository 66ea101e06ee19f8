/*
 * subpixel_oracle.c — CPU oracle of the sub-pixel refinement (include/usv_b200.h, usv_refine_subpixel_device).
 *
 * TEST INFRASTRUCTURE ONLY: tests/test_subpixel.py compiles it into a temporary directory and loads it with ctypes.
 * It includes the block-search oracle's source, so the candidate costs come from the same window_sums /
 * score_from_sums the dense parity suite checks the sweeps against. Build with -ffp-contract=off (as the oracle):
 * every f64 operation below is one correctly rounded IEEE operation, in the order the header states.
 */
#include "../oracle/block_search_oracle.c"

/* usv_oracle_distance at a fractional disparity (the refined distance) */
double usv_subpixel_oracle_distance_f64(double disp, int32_t kind) {
  switch (kind) {
    case USV_DIST_PINHOLE: return ((201.6 * 4) / (disp * 0.000043)) / 1000;
    case USV_DIST_POWERLAW: return pow(((10760 * pow(disp, -0.877)) / 3.0752), (1 / 0.7791));
    default: return 0.0;
  }
}

/*
 * The parabola through the costs of x*-1, x*, x*+1 in the sweep's terms (exact integer SAD / SSD, MatchValue 1 - score
 * for NCC / ZNCC), its vertex in 1/16 px rounded half away from zero, clamped to +-8; q = 0 unless both neighbours are
 * candidates of the window. right_index / out_x16 / out_dist: [n_pairs][ny*nx]; out_dist may be NULL.
 */
int usv_subpixel_oracle_refine(const uint8_t *left, const uint8_t *right, const usv_frame_desc *f, int32_t n_pairs,
                               const usv_search_params *p, const uint32_t *right_index, int32_t *out_x16,
                               double *out_dist) {
  int32_t nx, ny;
  if (usv_oracle_grid_dims(f, p, &nx, &ny, NULL)) return -1;
  const int nxc = f->width - p->tmpl_w + 1;
  const int64_t nwin = (int64_t)nx * ny, total = nwin * n_pairs;
  const int64_t n = (int64_t)p->tmpl_w * p->tmpl_h * f->channels;
  const int integer = p->cost_kind <= USV_COST_SSD;
#pragma omp parallel for schedule(dynamic, 256)
  for (int64_t g = 0; g < total; ++g) {
    const int64_t pr = g / nwin, w = g % nwin;
    const int x = (int)(w % nx) * p->stride_x, y = (int)(w / nx) * p->stride_y;
    const uint32_t r = right_index[g];
    int lo, hi;
    cand_range(x, nxc, p, &lo, &hi);
    const int xs = (int)(r % (uint32_t)nxc);
    int32_t x16 = USV_NO_SUBPIXEL;
    double dist = 0.0;
    if (r != USV_NO_MATCH && r / (uint32_t)nxc == (uint32_t)y && xs >= lo && xs <= hi) {
      const int d = p->camera_side == USV_LEFT_CAM ? x - xs : xs - x;
      int q = 0;
      if (xs - 1 >= lo && xs + 1 <= hi) {
        const uint8_t *L = left + (size_t)pr * f->frame_stride, *R = right + (size_t)pr * f->frame_stride;
        int64_t ci[3];
        double cv[3];
        for (int j = 0; j < 3; ++j) {
          usv_oracle_sums s;
          window_sums(L, R, f->row_stride, f->channels, x, xs - 1 + j, y, p->tmpl_w, p->tmpl_h, p->cost_kind, &s);
          ci[j] = p->cost_kind == USV_COST_SAD ? (int64_t)s.sad : (int64_t)s.ssd;
          cv[j] = integer ? 0.0 : 1.0 - score_from_sums(&s, n, p->cost_kind);
        }
        if (integer) {
          const int64_t num = ci[0] - ci[2], den = ci[0] + ci[2] - 2 * ci[1];
          if (den > 0) {
            int64_t m = (16 * (num < 0 ? -num : num) + den) / (2 * den);
            if (m > 8) m = 8;
            q = (int)(num < 0 ? -m : m);
          }
        } else {
          const double num = cv[0] - cv[2], den = (cv[0] - cv[1]) + (cv[2] - cv[1]);
          if (den > 0) {
            double t = round(8.0 * num / den);
            q = (int)(t > 8.0 ? 8.0 : t < -8.0 ? -8.0 : t);
          }
        }
      }
      x16 = p->camera_side == USV_LEFT_CAM ? 16 * d - q : 16 * d + q;
      dist = usv_subpixel_oracle_distance_f64(x16 / 16.0, p->distance_kind);
    }
    out_x16[g] = x16;
    if (out_dist) out_dist[g] = dist;
  }
  return 0;
}
