// usv_host_test.cpp — exercises the C++ drop-in interfaces (Match / SearchAlgorithms /
// DistanceCalculator) the way the reference's call sites use them (P/Main.cpp:1115-1143,
// :1238-1247), checks the reference's known answers (SURVEY.md section 4) and dumps the frames
// and results so that tests/test_host_cpp.py can compare them with the CPU oracle.
//   usv_host_test <dump-file>
//   usv_host_test --bench <pairs> <n_devices> <steps> <warmup>     (one JSON line: the C++ drop-in's throughput)
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <vector>

#include "SearchAlgorithms.hpp"

static int fails = 0;
#define CHECK(cond)                                                        \
  do {                                                                     \
    if (!(cond)) { std::printf("FAIL %s:%d: %s\n", __FILE__, __LINE__, #cond); ++fails; } \
  } while (0)

static bool close_rel(double a, double b, double rel) { return std::fabs(a - b) <= rel * std::fabs(b); }

// Throughput of the C++ layer on the bench workload (640x480 gray, 16x16 SAD, full range): BlockSearchBatch over
// n_dev GPUs (one worker thread + context + pinned ring per GPU, results into disjoint slices of one pinned host
// array) and the per-pair BlockSearch call of the reference's call sites. Host buffers, copies both ways timed.
static int run_bench(int pairs, int n_dev, int steps, int warmup) {
  const int W = 640, H = 480;
  const size_t fsz = (size_t)W * H;
  std::vector<uint8_t> L(fsz * pairs), R(fsz * pairs);
  uint32_t s = 325u;
  auto rnd = [&]() { s = s * 1664525u + 1013904223u; return (uint8_t)(s >> 24); };
  for (int p = 0; p < pairs; ++p) {
    uint8_t* l = L.data() + fsz * p;
    uint8_t* r = R.data() + fsz * p;
    for (size_t k = 0; k < fsz; ++k) l[k] = rnd();
    for (int y = 0; y < H; ++y)
      for (int x = 0; x < W; ++x) r[(size_t)y * W + x] = x + 37 < W ? l[(size_t)y * W + x + 37] : rnd();
  }
  BlockSearchSpec spec;
  const size_t n_win = (size_t)(W - 15) * (H - 15);
  std::vector<unsigned short> disp(n_win * pairs), cost(n_win * pairs);
  std::vector<int> devices;
  for (int g = 0; g < n_dev; ++g) devices.push_back(g);
  if (BlockSearchPinHostBuffer(L.data(), L.size()) || BlockSearchPinHostBuffer(R.data(), R.size()) ||
      BlockSearchPinHostBuffer(disp.data(), disp.size() * 2) || BlockSearchPinHostBuffer(cost.data(), cost.size() * 2)) {
    std::printf("{\"error\": \"%s\"}\n", BlockSearchLastError());
    return 2;
  }
  BlockSearchBatchStats st;
  auto run = [&](unsigned short* cost_out) { return BlockSearchBatch(L.data(), R.data(), pairs, W, H, W, fsz, spec, devices, disp.data(), cost_out, &st); };
  double t_disp = 0.0, t_both = 0.0;
  for (int variant = 0; variant < 2; ++variant) {
    unsigned short* co = variant ? cost.data() : nullptr;
    for (int k = 0; k < warmup; ++k)
      if (run(co)) { std::printf("{\"error\": \"%s\"}\n", BlockSearchLastError()); return 2; }
    const auto t0 = std::chrono::steady_clock::now();
    for (int k = 0; k < steps; ++k) run(co);
    (variant ? t_both : t_disp) = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  }
  // sanity of the timed output: the known shift is recovered, at cost 0
  size_t good = 0, seen = 0;
  for (int p = 0; p < pairs; p += std::max(1, pairs / 4))
    for (int y = 0; y < H - 15; y += 29)
      for (int x = 37; x < W - 15; x += 7) { ++seen; good += disp[(size_t)p * n_win + (size_t)y * (W - 15) + x] == 37 && cost[(size_t)p * n_win + (size_t)y * (W - 15) + x] == 0; }
  // the reference-shaped per-pair call (generate -> resolve -> distance, vectors out)
  usv::ImageView left(L.data(), W, H, 1, W), right(R.data(), W, H, 1, W);
  std::vector<Match> m;
  std::vector<double> d;
  int n_single = 0;
  for (int k = 0; k < 3; ++k) BlockSearch(LeftCam, &left, &right, spec, m, d);
  const auto t1 = std::chrono::steady_clock::now();
  double t_single = 0.0;
  while (t_single < 1.0) {
    usv::ImageView l2(L.data() + fsz * (n_single % pairs), W, H, 1, W), r2(R.data() + fsz * (n_single % pairs), W, H, 1, W);
    BlockSearch(LeftCam, &l2, &r2, spec, m, d);
    ++n_single;
    t_single = std::chrono::duration<double>(std::chrono::steady_clock::now() - t1).count();
  }
  std::printf("{\"api\": \"BlockSearchBatch (C++), one worker thread + context + pinned ring per GPU, frames from and results into the caller's "
              "page-locked arrays\", \"pairs\": %d, \"n_devices\": %d, \"steps\": %d, \"pairs_per_s\": %.1f, \"outputs\": \"resolved_disparity_u16 (2 B/window)\", "
              "\"with_cost\": {\"pairs_per_s\": %.1f, \"outputs\": \"resolved_disparity_u16 + raw_cost_u16 (4 B/window)\"}, "
              "\"known_shift_recovered\": %s, \"block_search_single_pair\": {\"api\": \"BlockSearch (generate -> resolve -> distance, std::vector<Match> out), one "
              "host thread\", \"pairs_per_s\": %.1f, \"matches_per_pair\": %zu}}\n",
              pairs, n_dev, steps, (double)pairs * steps / t_disp, (double)pairs * steps / t_both, good == seen ? "true" : "false", n_single / t_single, m.size());
  BlockSearchUnpinHostBuffer(L.data());
  BlockSearchUnpinHostBuffer(R.data());
  BlockSearchUnpinHostBuffer(disp.data());
  BlockSearchUnpinHostBuffer(cost.data());
  return good == seen ? 0 : 1;
}

int main(int argc, char** argv) {
  if (argc >= 6 && std::strcmp(argv[1], "--bench") == 0) return run_bench(std::atoi(argv[2]), std::atoi(argv[3]), std::atoi(argv[4]), std::atoi(argv[5]));
  // ---- Match: the reference's record
  static_assert(sizeof(Match) == 16, "Match layout");
  Match m0(1, 2, 0.5);
  CHECK(m0.LeftIndex == 1 && m0.RightIndex == 2 && m0.MatchValue == 0.5);

  // ---- ResolveMatchList known answers (reference code, SURVEY.md section 4)
  {
    std::vector<Match> in = {{0, 0, .5}, {0, 1, .3}, {0, 2, .4}, {0, 3, .1}, {0, 4, .2}}, out;
    ResolveMatchList(in, out);
    CHECK(out.size() == 3 && out[0].RightIndex == 3 && out[1].RightIndex == 3 && out[2].RightIndex == 4);
    in = {{0, 0, .3}, {0, 1, .3}, {0, 2, .5}};
    ResolveMatchList(in, out);
    CHECK(out.size() == 3 && out[0].RightIndex == 0 && out[1].RightIndex == 1);  // equal later candidate never replaces
    in = {{0, 0, .5}, {1, 1, .6}, {0, 1, .1}};
    ResolveMatchList(in, out);
    CHECK(out.size() == 2 && out[0].LeftIndex == 0 && out[0].RightIndex == 1 && out[1].RightIndex == 1);
  }

  // ---- the reference's original call (P/Main.cpp:1115-1117): contour lists in, Match list out
  {
    std::vector<std::vector<cv::Point> > Lc = {{{10, 10}, {60, 10}, {60, 40}, {10, 40}}, {{100, 100}, {130, 160}, {70, 160}}};
    std::vector<std::vector<cv::Point> > Rc = {{{5, 12}, {54, 12}, {54, 43}, {5, 43}}, {{90, 100}, {121, 158}, {60, 161}}, {{0, 0}, {200, 0}, {200, 5}}};
    std::vector<Match> Matcher, Tentative;
    GenerateMatchingList(Lc, Rc, Matcher);
    CHECK(Matcher.size() >= 2);
    ResolveMatchList(Matcher, Tentative);
    bool rect_ok = false, tri_ok = false;
    for (const Match& m : Tentative) { rect_ok |= (m.LeftIndex == 0 && m.RightIndex == 0); tri_ok |= (m.LeftIndex == 1 && m.RightIndex == 1); }
    CHECK(rect_ok && tri_ok);  // the rectangle pairs with the rectangle, the triangle with the triangle
    std::vector<Match> none;
    GenerateMatchingList(Lc, std::vector<std::vector<cv::Point> >(), none);
    CHECK(none.empty());  // :405
  }

  // ---- IDMatcher: the reference's join, comma-operator quirk included (P/Main.cpp:492)
  {
    std::vector<Match> cur = {{0, 5, .1}, {1, 7, .2}, {2, 5, .3}}, old = {{5, 9, .1}, {7, 3, .2}, {8, 1, .3}};
    std::vector<cv::Point3i> c;
    IDMatcher(cur, old, c);
    CHECK(c.size() == 3 && c[0].x == 9 && c[0].y == 0 && c[0].z == 0 && c[1].x == 3 && c[2].x == 9);
  }

  // ---- synthetic rectified pair: right[y][x] = left[y][x + 37]
  const int W = 640, H = 64, SHIFT = 37;
  std::vector<uint8_t> L((size_t)W * H), R((size_t)W * H);
  uint32_t s = 325u;
  auto rnd = [&]() { s = s * 1664525u + 1013904223u; return (uint8_t)(s >> 24); };
  for (auto& v : L) v = rnd();
  for (int y = 0; y < H; ++y)
    for (int x = 0; x < W; ++x) R[(size_t)y * W + x] = x + SHIFT < W ? L[(size_t)y * W + x + SHIFT] : rnd();
  usv::ImageView left(L.data(), W, H, 1, W), right(R.data(), W, H, 1, W);

  // ---- the reference's call order: generate -> resolve -> distance, in one call
  BlockSearchSpec spec;
  std::vector<Match> matches;
  std::vector<double> dist;
  int rc = BlockSearch(LeftCam, &left, &right, spec, matches, dist);
  if (rc != 0) { std::printf("BlockSearch failed: %s\n", BlockSearchLastError()); return 2; }
  const int nxc = W - 16 + 1, nyc = H - 16 + 1;
  CHECK(matches.size() == dist.size() && !matches.empty());
  // BlockSearch = ResolveMatchList over the accepted per-window winners: a window with an exact counterpart (cost 0) is never
  // strictly beaten, so every such window is in the list (possibly more than once: the reference keeps duplicates)
  std::vector<char> seen_exact((size_t)nxc * nyc, 0);
  size_t exact = 0;
  for (size_t k = 0; k < matches.size(); ++k) {
    const int x = matches[k].LeftIndex % nxc, y = matches[k].LeftIndex / nxc, xr = matches[k].RightIndex - y * nxc;
    if (x >= SHIFT) { CHECK(x - xr == SHIFT && matches[k].MatchValue == 0.0); if (!seen_exact[matches[k].LeftIndex]) { seen_exact[matches[k].LeftIndex] = 1; ++exact; } }
    CHECK(close_rel(dist[k], ((201.6 * 4) / ((x - xr) * 0.000043)) / 1000, 1e-12) || x == xr);
  }
  CHECK(exact == (size_t)(nxc - SHIFT) * nyc);
  // the batch form over the same pair: the resolved disparity map marks exactly the windows that appear in the list
  {
    std::vector<unsigned short> rd((size_t)nxc * nyc), rc16((size_t)nxc * nyc);
    BlockSearchBatchStats bs;
    CHECK(BlockSearchBatch(L.data(), R.data(), 1, W, H, W, (size_t)W * H, spec, std::vector<int>{0}, rd.data(), rc16.data(), &bs) == 0);
    std::vector<char> in_list((size_t)nxc * nyc, 0);
    for (const Match& m : matches) in_list[m.LeftIndex] = 1;
    size_t bad = 0;
    for (size_t w = 0; w < rd.size(); ++w) bad += (rd[w] != 0xFFFF) != (in_list[w] != 0);
    CHECK(bad == 0 && bs.DevicesUsed == 1 && bs.PairsPerDevice[0] == 1);
    std::vector<double> table;
    CHECK(DistanceTable(spec, W, table) == 0 && table.size() == (size_t)W);
    for (size_t k = 0; k < matches.size(); k += 97) CHECK(table[rd[matches[k].LeftIndex]] == dist[k]);
  }
  CHECK(BlockSearch(LeftCam, nullptr, &right, spec, matches, dist) == -1);  // empty frame -> -1 (P/Main.cpp:908-911)
  rc = BlockSearch(LeftCam, &left, &right, spec, matches, dist);
  CHECK(rc == 0);

  // ---- explicit templates: the full candidate list, then the reference's resolve
  std::vector<Match> all, tentative;
  BlockSearchSpec zs = spec;
  zs.Cost = BlockSearchSpec::ZNCC;
  zs.AcceptThreshold = 0.75;
  GenerateMatchingList(left, right, std::vector<cv::Point>{{300, 20}, {400, 30}}, zs, all);
  CHECK(!all.empty());
  ResolveMatchList(all, tentative);
  CHECK(!tentative.empty() && tentative[0].LeftIndex == 0 && tentative[0].RightIndex == 20u * nxc + (300 - SHIFT));
  for (size_t k = 1; k < all.size(); ++k)  // i-major, j-minor order (P/Main.cpp:408-410)
    CHECK(all[k - 1].LeftIndex < all[k].LeftIndex || (all[k - 1].LeftIndex == all[k].LeftIndex && all[k - 1].RightIndex < all[k].RightIndex));

  // ---- pre-pass: gray of a BGR frame, both arithmetic flavours (P/Main.cpp:921; 14-bit vs 15-bit coefficients)
  {
    std::vector<uint8_t> bgr(3 * 8 * 4), g3(8 * 4), g4(8 * 4);
    for (size_t k = 0; k < bgr.size(); ++k) bgr[k] = (uint8_t)(37 * k + 11);
    usv::ImageView v(bgr.data(), 8, 4, 3, 24);
    CHECK(RectifyLightingGray(v, nullptr, nullptr, false, g3.data(), 8, true) == 0);
    CHECK(RectifyLightingGray(v, nullptr, nullptr, false, g4.data(), 8, false) == 0);
    for (int k = 0; k < 32; ++k) {
      const int b = bgr[3 * k], g = bgr[3 * k + 1], r = bgr[3 * k + 2];
      CHECK(g3[k] == ((b * 1868 + g * 9617 + r * 4899 + (1 << 13)) >> 14));
      CHECK(g4[k] == ((b * 3735 + g * 19235 + r * 9798 + (1 << 14)) >> 15));
    }
  }
  // ---- pre-pass on ROIs (a cv::Mat window: step > row bytes): the source is a 13x7 window of a 23x11 BGR image, the
  // output a 13x7 window of a 31x11 gray image. Every gray pixel outside the output window keeps its value; with lighting
  // off the window holds the gray formula of the source window.
  {
    const int IW = 23, IH = 11, GW = 31, RW = 13, RH = 7, X0 = 5, Y0 = 2;  // odd width and step: the byte-store path
    const uint8_t kSentinel = 0xA5;
    std::vector<uint8_t> img(3 * IW * IH), gray(GW * IH);
    for (size_t k = 0; k < img.size(); ++k) img[k] = (uint8_t)(53 * k + 7);
    usv::ImageView roi(img.data() + (size_t)Y0 * 3 * IW + 3 * X0, RW, RH, 3, 3 * IW);
    for (int lighting = 0; lighting < 2; ++lighting) {
      for (int opencv3 = 0; opencv3 < 2; ++opencv3) {
        std::fill(gray.begin(), gray.end(), kSentinel);
        CHECK(RectifyLightingGray(roi, nullptr, nullptr, lighting != 0, gray.data() + (size_t)Y0 * GW + X0, GW, opencv3 != 0) == 0);
        int outside_changed = 0, inside_wrong = 0;
        for (int y = 0; y < IH; ++y)
          for (int x = 0; x < GW; ++x) {
            const bool in = y >= Y0 && y < Y0 + RH && x >= X0 && x < X0 + RW;
            const uint8_t got = gray[(size_t)y * GW + x];
            if (!in) { outside_changed += got != kSentinel; continue; }
            if (lighting) continue;
            const uint8_t* px = img.data() + (size_t)y * 3 * IW + 3 * x;
            const int b = px[0], g = px[1], r = px[2];
            inside_wrong += got != (opencv3 ? (b * 1868 + g * 9617 + r * 4899 + (1 << 13)) >> 14
                                            : (b * 3735 + g * 19235 + r * 9798 + (1 << 14)) >> 15);
          }
        CHECK(outside_changed == 0);
        CHECK(inside_wrong == 0);
      }
    }
  }

  // ---- DistanceCalculator known answers (reference code, SURVEY.md section 4)
  {
    using tp = std::chrono::steady_clock::time_point;
    auto ms = [](int v) { return tp(std::chrono::duration_cast<std::chrono::steady_clock::duration>(std::chrono::milliseconds(v))); };
    std::vector<double> d;
    MovingObjectDistanceCalculator(LeftCam, ms(110), {{300, 200}}, {{260, 200}}, {{250, 200}}, {{240, 200}}, {}, {{0, 0, 0}}, ms(100),
                                   ms(67), ms(33), d);
    CHECK(d.size() == 1 && close_rel(d[0], 626.463714398, 1e-10));
    d.clear();
    MovingObjectDistanceCalculator(LeftCam, ms(110), {{300, 200}}, {}, {{250, 200}}, {{240, 200}}, {}, {{0, 0, 0}}, ms(100), ms(67),
                                   ms(33), d);
    CHECK(d.empty());  // an empty other-camera history produces nothing (:28)
    std::vector<cv::Point3d> pos;
    CooridinatePositionCalculator(LeftCam, {100.0}, {{300, 200}}, pos);
    CHECK(pos.empty());  // gated by the UI flag (:92)
    CoordinateDisplay = true;
    CooridinatePositionCalculator(LeftCam, {100.0}, {{300, 200}}, pos);
    CooridinatePositionCalculator(RightCam, {100.0}, {{300, 200}}, pos);
    CHECK(pos.size() == 2 && std::fabs(pos[0].x - 9.103702) < 1e-6 && std::fabs(pos[0].y - 99.584751) < 1e-6 &&
          std::fabs(pos[0].z - 12.454575) < 1e-6 && std::fabs(pos[1].x + 18.505677) < 1e-6);
    std::vector<double> dd;
    DisparityToDistance({40, 0, 64}, true, dd);
    CHECK(dd.size() == 3 && close_rel(dd[0], 556.401951467, 1e-10) && std::isinf(dd[1]) && close_rel(dd[2], 327.8079, 1e-6));
    CHECK(deg2rad(180.0) == 180.0 * PI / 180.0 && rad2deg(1.0) == 1.0 * 180 / PI);
  }

  // ---- re-entrancy: the reference calls these from four threads at once (SURVEY.md 8b)
  {
    std::vector<std::vector<Match>> res(4);
    std::vector<std::thread> th;
    for (int t = 0; t < 4; ++t)
      th.emplace_back([&, t]() {
        std::vector<double> dd;
        BlockSearch(LeftCam, &left, &right, spec, res[t], dd);
      });
    for (auto& t : th) t.join();
    for (int t = 1; t < 4; ++t)
      CHECK(res[t].size() == res[0].size() && std::memcmp(res[t].data(), res[0].data(), res[0].size() * sizeof(Match)) == 0);
  }

  // ---- dump for the oracle cross-check in pytest
  if (argc > 1) {
    FILE* f = std::fopen(argv[1], "wb");
    if (!f) { std::printf("cannot write %s\n", argv[1]); return 3; }
    const int32_t hdr[4] = {W, H, (int32_t)matches.size(), (int32_t)all.size()};
    std::fwrite(hdr, sizeof(hdr), 1, f);
    std::fwrite(L.data(), 1, L.size(), f);
    std::fwrite(R.data(), 1, R.size(), f);
    std::fwrite(matches.data(), sizeof(Match), matches.size(), f);
    std::fwrite(dist.data(), sizeof(double), dist.size(), f);
    std::fwrite(all.data(), sizeof(Match), all.size(), f);
    std::fclose(f);
  }
  std::printf("%s (%d failures, %zu dense matches, %zu template candidates)\n", fails ? "FAILED" : "PASSED", fails, matches.size(),
              all.size());
  return fails ? 1 : 0;
}
