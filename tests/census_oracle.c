/*
 * census_oracle.c — CPU oracle of USV_COST_CENSUS (include/usv_b200.h), for tests/test_census.py.
 *
 * TEST INFRASTRUCTURE ONLY. Direct form on purpose, and a different formulation from the library's: the census byte of
 * every template and candidate pixel is computed on the fly from the frame, with the border rule, and the window cost is
 * the sum of per-byte popcounts. The rest (candidate enumeration, first minimum, accept test, indices, disparity,
 * distance) restates oracle/block_search_oracle.c:match_one for an integer cost:
 *   - candidates in ascending x' (P/Main.cpp:410), an equal later candidate never replaces (P/Main.cpp:451)
 *   - accept `MatchValue < threshold` (P/Main.cpp:417), MatchValue = H / (8 n)
 *   - disparity by camera side (P/Main.cpp:681-693), pinhole (P/Main.cpp:694) and power-law
 *     (P/DistanceCalculator.cpp:84) distance
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

#include "../include/usv_b200.h"

/* census byte of pixel (x, y), channel c */
static inline uint8_t census_at(const uint8_t *F, int rs, int W, int H, int C, int x, int y, int c) {
  static const int dx[8] = {-1, 0, 1, -1, 1, -1, 0, 1}, dy[8] = {-1, -1, -1, 0, 0, 1, 1, 1};
  const int v = F[(size_t)y * rs + (size_t)x * C + c];
  uint8_t out = 0;
  for (int k = 0; k < 8; ++k) {
    const int nx = x + dx[k], ny = y + dy[k];
    if (nx < 0 || nx >= W || ny < 0 || ny >= H) continue;
    if (F[(size_t)ny * rs + (size_t)nx * C + c] < v) out |= (uint8_t)(1u << k);
  }
  return out;
}

static inline uint32_t window_hamming(const uint8_t *L, const uint8_t *R, const usv_frame_desc *f, int lx, int rx, int y,
                                      int tw, int th) {
  uint32_t h = 0;
  for (int dy = 0; dy < th; ++dy)
    for (int dx = 0; dx < tw; ++dx)
      for (int c = 0; c < f->channels; ++c) {
        const uint8_t a = census_at(L, f->row_stride, f->width, f->height, f->channels, lx + dx, y + dy, c);
        const uint8_t b = census_at(R, f->row_stride, f->width, f->height, f->channels, rx + dx, y + dy, c);
        h += (uint32_t)__builtin_popcount((unsigned)(a ^ b));
      }
  return h;
}

double usv_census_oracle_distance(int32_t disp, int32_t kind) {
  switch (kind) {
    case USV_DIST_PINHOLE: return ((201.6 * 4) / (disp * 0.000043)) / 1000;
    case USV_DIST_POWERLAW: return pow(((10760 * pow(disp, -0.877)) / 3.0752), (1 / 0.7791));
    default: return 0.0;
  }
}

static void match_one(const uint8_t *L, const uint8_t *R, const usv_frame_desc *f, const usv_search_params *p, int x, int y,
                      uint32_t left_index, const usv_outputs *o, int64_t g, uint32_t *cost_row) {
  const int nxc = f->width - p->tmpl_w + 1;
  const int64_t n = (int64_t)p->tmpl_w * p->tmpl_h * f->channels;
  int lo, hi;
  if (p->camera_side == USV_LEFT_CAM) { lo = x - p->search_max; hi = x - p->search_min; }
  else { lo = x + p->search_min; hi = x + p->search_max; }
  if (lo < 0) lo = 0;
  if (hi > nxc - 1) hi = nxc - 1;
  uint32_t best = 0xFFFFFFFFu;
  int best_x = -1;
  for (int xr = lo; xr <= hi; ++xr) {
    const uint32_t h = window_hamming(L, R, f, x, xr, y, p->tmpl_w, p->tmpl_h);
    if (cost_row) cost_row[xr - lo] = h;
    if (best_x < 0 || h < best) { best = h; best_x = xr; }
  }
  const double v = best_x >= 0 ? (double)best / (double)(8 * n) : INFINITY;
  const int accepted = best_x >= 0 && v < p->accept_threshold;
  const int d = best_x >= 0 ? (p->camera_side == USV_LEFT_CAM ? x - best_x : best_x - x) : 0;
  const uint32_t rindex = accepted ? (uint32_t)(y * nxc + best_x) : USV_NO_MATCH;
  const double dd = accepted ? usv_census_oracle_distance(d, p->distance_kind) : 0.0;
  if (o->matches) { o->matches[g].LeftIndex = left_index; o->matches[g].RightIndex = rindex; o->matches[g].MatchValue = v; }
  if (o->right_index) o->right_index[g] = rindex;
  if (o->raw_cost) o->raw_cost[g] = best;
  if (o->raw_cost_u16) o->raw_cost_u16[g] = (uint16_t)best;
  if (o->score) o->score[g] = 0.0;
  if (o->distance) o->distance[g] = dd;
  if (o->distance_f32) o->distance_f32[g] = (float)dd;
  if (o->disparity_u16) o->disparity_u16[g] = accepted ? (uint16_t)d : (uint16_t)USV_NO_DISPARITY;
}

/* every window of the grid x = ix * stride_x, y = iy * stride_y, outputs [pair][iy * nx + ix] */
int usv_census_oracle_match_dense(const uint8_t *left, const uint8_t *right, const usv_frame_desc *f, int32_t n_pairs,
                                  const usv_search_params *p, const usv_outputs *o) {
  const int nxc = f->width - p->tmpl_w + 1, nyc = f->height - p->tmpl_h + 1;
  if (nxc <= 0 || nyc <= 0 || p->stride_x <= 0 || p->stride_y <= 0) return -1;
  const int nx = (nxc - 1) / p->stride_x + 1, ny = (nyc - 1) / p->stride_y + 1;
  for (int32_t pr = 0; pr < n_pairs; ++pr) {
    const uint8_t *L = left + (size_t)pr * f->frame_stride, *R = right + (size_t)pr * f->frame_stride;
#pragma omp parallel for schedule(dynamic, 1)
    for (int iy = 0; iy < ny; ++iy)
      for (int ix = 0; ix < nx; ++ix) {
        const int64_t w = (int64_t)iy * nx + ix;
        match_one(L, R, f, p, ix * p->stride_x, iy * p->stride_y, (uint32_t)w, o, (int64_t)pr * nx * ny + w, NULL);
      }
  }
  return 0;
}

/* a template list shared by all pairs; cost_rows (optional): [pair][template][row_cap], every candidate's H in scan order */
int usv_census_oracle_match_templates(const uint8_t *left, const uint8_t *right, const usv_frame_desc *f, int32_t n_pairs,
                                      const int32_t *tx, const int32_t *ty, int32_t n_templates, const usv_search_params *p,
                                      const usv_outputs *o, uint32_t *cost_rows, int32_t row_cap) {
  const int nxc = f->width - p->tmpl_w + 1, nyc = f->height - p->tmpl_h + 1;
  if (nxc <= 0 || nyc <= 0 || row_cap < f->width) return -1;
  for (int32_t pr = 0; pr < n_pairs; ++pr) {
    const uint8_t *L = left + (size_t)pr * f->frame_stride, *R = right + (size_t)pr * f->frame_stride;
    for (int t = 0; t < n_templates; ++t) {
      if (tx[t] < 0 || tx[t] >= nxc || ty[t] < 0 || ty[t] >= nyc) return -1;
      const int64_t g = (int64_t)pr * n_templates + t;
      match_one(L, R, f, p, tx[t], ty[t], (uint32_t)t, o, g, cost_rows ? cost_rows + g * row_cap : NULL);
    }
  }
  return 0;
}
