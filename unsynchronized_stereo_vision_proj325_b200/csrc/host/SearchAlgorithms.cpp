// SearchAlgorithms.cpp — host side of the block-search drop-in. Every cost is computed by the
// sm_100a kernels behind the C-ABI; this file only marshals vectors, applies the accept test to
// dumped candidate costs (template overload) and forwards ResolveMatchList to the GPU resolve.
#include "../../../include/SearchAlgorithms.hpp"

#include <chrono>
#include <cmath>
#include <cstring>
#include <map>
#include <mutex>
#include <thread>

#include "usv_host_ctx.hpp"

static usv_search_params to_params(const BlockSearchSpec& s) {
  usv_search_params p;
  std::memset(&p, 0, sizeof(p));
  p.tmpl_w = s.TemplateWidth; p.tmpl_h = s.TemplateHeight;
  p.search_min = s.SearchMin; p.search_max = s.SearchMax;
  p.stride_x = s.StrideX; p.stride_y = s.StrideY;
  p.cost_kind = (int)s.Cost;
  p.camera_side = s.CameraSide == LeftCam ? USV_LEFT_CAM : USV_RIGHT_CAM;
  p.distance_kind = (int)s.Distance;
  p.accept_threshold = s.AcceptThreshold;
  return p;
}

static bool same_geometry(const usv::ImageView& a, const usv::ImageView& b) {
  return a.data && b.data && a.width == b.width && a.height == b.height && a.channels == b.channels && a.step == b.step;
}

static usv_frame_desc to_frame(const usv::ImageView& v) {
  usv_frame_desc f;
  f.width = v.width; f.height = v.height; f.channels = v.channels;
  f.row_stride = (int32_t)v.step;
  f.frame_stride = (int64_t)v.step * v.height;
  return f;
}

const char* BlockSearchLastError() { return usv::thread_contexts().last_error.c_str(); }

// P/Main.cpp:403-426, original arguments: the all-pairs shape + size cost runs in usv_contours.cu
void GenerateMatchingList(std::vector<std::vector<cv::Point> > UsefulContoursL, std::vector<std::vector<cv::Point> > UsefulContoursR,
                          std::vector<Match>& Matcher) {
  if (UsefulContoursL.empty() || UsefulContoursR.empty()) return;  // :405
  usv::ThreadContexts& tc = usv::thread_contexts();
  usv_ctx* ctx = tc.get(0);
  if (!ctx) return;
  auto pack = [](const std::vector<std::vector<cv::Point> >& cs, std::vector<int32_t>& pts, std::vector<int32_t>& off) {
    off.assign(1, 0);
    for (const auto& c : cs) {
      for (const auto& p : c) { pts.push_back(p.x); pts.push_back(p.y); }
      off.push_back((int32_t)(pts.size() / 2));
    }
    if (pts.empty()) pts.resize(2, 0);
  };
  std::vector<int32_t> pl, ol, pr, orr;
  pack(UsefulContoursL, pl, ol);
  pack(UsefulContoursR, pr, orr);
  std::vector<usv_match> out(UsefulContoursL.size() * UsefulContoursR.size());
  int64_t n = 0;
  const int rc = usv_match_contours(ctx, pl.data(), ol.data(), (int32_t)UsefulContoursL.size(), pr.data(), orr.data(),
                                    (int32_t)UsefulContoursR.size(), 0.75 /* :417 */, out.data(), (int64_t)out.size(), &n, nullptr);
  if (!tc.check(ctx, rc, "usv_match_contours")) return;
  for (int64_t k = 0; k < n; ++k) Matcher.push_back({out[k].LeftIndex, out[k].RightIndex, out[k].MatchValue});  // :418
}

void GenerateMatchingList(const usv::ImageView& ThisCamera, const usv::ImageView& OtherCamera, const BlockSearchSpec& Spec,
                          std::vector<Match>& Matcher, std::vector<double>* Distances) {
  usv::ThreadContexts& tc = usv::thread_contexts();
  if (!same_geometry(ThisCamera, OtherCamera)) { tc.last_error = "GenerateMatchingList: frames empty or of different geometry"; return; }
  usv_ctx* ctx = tc.get(Spec.Device);
  if (!ctx) return;
  const usv_search_params p = to_params(Spec);
  const usv_frame_desc f = to_frame(ThisCamera);
  int32_t nx = 0, ny = 0;
  if (usv_grid_dims(&f, &p, &nx, &ny, nullptr) != USV_OK) { tc.last_error = "GenerateMatchingList: template does not fit the frame"; return; }
  const size_t n = (size_t)nx * ny;
  // thread-local result buffers, reused from call to call (no 4.6 MB allocation + page faults per frame pair)
  static thread_local std::vector<usv_match> rec;
  static thread_local std::vector<double> dist;
  if (rec.size() < n) rec.resize(n);
  if (Distances && dist.size() < n) dist.resize(n);
  usv_outputs out;
  std::memset(&out, 0, sizeof(out));
  out.matches = rec.data();
  if (Distances) out.distance = dist.data();
  const int rc = usv_match_dense_host(ctx, ThisCamera.data, OtherCamera.data, &f, 1, &p, &out);
  if (!tc.check(ctx, rc, "usv_match_dense_host")) return;
  static_assert(sizeof(Match) == sizeof(usv_match), "Match must stay bit-identical to usv_match");
  const Match* as_match = reinterpret_cast<const Match*>(rec.data());
  // runs of accepted windows are appended in bulk (usually the whole list is one run)
  for (size_t i = 0; i < n;) {
    if (rec[i].RightIndex == USV_NO_MATCH) { ++i; continue; }  // no candidate passed `< AcceptThreshold` (P/Main.cpp:417)
    size_t j = i + 1;
    while (j < n && rec[j].RightIndex != USV_NO_MATCH) ++j;
    Matcher.insert(Matcher.end(), as_match + i, as_match + j);
    if (Distances) Distances->insert(Distances->end(), dist.begin() + i, dist.begin() + j);
    i = j;
  }
}

void GenerateMatchingList(const usv::ImageView& ThisCamera, const usv::ImageView& OtherCamera, std::vector<cv::Point> Templates,
                          const BlockSearchSpec& Spec, std::vector<Match>& Matcher) {
  usv::ThreadContexts& tc = usv::thread_contexts();
  if (!same_geometry(ThisCamera, OtherCamera)) { tc.last_error = "GenerateMatchingList: frames empty or of different geometry"; return; }
  if (Templates.empty()) return;  // P/Main.cpp:405
  usv_ctx* ctx = tc.get(Spec.Device);
  if (!ctx) return;
  const usv_search_params p = to_params(Spec);
  const usv_frame_desc f = to_frame(ThisCamera);
  const int nt = (int)Templates.size(), cap = f.width;
  std::vector<int32_t> tx(nt), ty(nt);
  for (int i = 0; i < nt; ++i) { tx[i] = Templates[i].x; ty[i] = Templates[i].y; }
  const bool integer = p.cost_kind != USV_COST_NCC && p.cost_kind != USV_COST_ZNCC;
  std::vector<uint32_t> cost_rows(integer ? (size_t)nt * cap : 0);
  std::vector<double> score_rows(integer ? 0 : (size_t)nt * cap);
  usv_outputs out;
  std::memset(&out, 0, sizeof(out));
  const int rc = usv_match_templates_host(ctx, ThisCamera.data, OtherCamera.data, &f, 1, tx.data(), ty.data(), nt, &p, &out,
                                          integer ? cost_rows.data() : nullptr, integer ? nullptr : score_rows.data(), cap);
  if (!tc.check(ctx, rc, "usv_match_templates_host")) return;
  const int nxc = f.width - p.tmpl_w + 1;
  const double n_elems = (double)p.tmpl_w * p.tmpl_h * f.channels;
  const double den = (p.cost_kind == USV_COST_SAD ? 255.0 : p.cost_kind == USV_COST_CENSUS ? 8.0 : 65025.0) * n_elems;
  for (int i = 0; i < nt; ++i) {  // template-major (P/Main.cpp:408)
    int lo, hi;
    if (p.camera_side == USV_LEFT_CAM) { lo = tx[i] - p.search_max; hi = tx[i] - p.search_min; }
    else { lo = tx[i] + p.search_min; hi = tx[i] + p.search_max; }
    if (lo < 0) lo = 0;
    if (hi > nxc - 1) hi = nxc - 1;
    for (int xr = lo; xr <= hi; ++xr) {  // candidate-minor, ascending x' (P/Main.cpp:410)
      const size_t k = (size_t)i * cap + (xr - lo);
      const double v = integer ? (double)cost_rows[k] / den : 1.0 - score_rows[k];
      if (v < Spec.AcceptThreshold)  // Is it at least a partial match? (P/Main.cpp:417)
        Matcher.push_back({(unsigned)i, (unsigned)(ty[i] * nxc + xr), v});
    }
  }
}

// P/Main.cpp:432-477 behind the original signature. The greedy pass runs on the GPU (usv_resolve.cu: it factors
// into next-strictly-smaller chains per LeftIndex / RightIndex group, so lists of any length resolve in
// O(M log M)); the output is the reference's TentativeMatch entry for entry, duplicates included.
void ResolveMatchList(std::vector<Match> Matcher, std::vector<Match>& TentativeMatch) {
  TentativeMatch.clear();  // :437
  if (Matcher.empty()) return;  // :441
  usv::ThreadContexts& tc = usv::thread_contexts();
  usv_ctx* ctx = tc.get(0);
  if (!ctx) return;
  static_assert(sizeof(Match) == sizeof(usv_match), "Match must stay bit-identical to usv_match");
  std::vector<usv_match> out(Matcher.size());
  int64_t n = 0;
  const int rc = usv_resolve_match_list(ctx, reinterpret_cast<const usv_match*>(Matcher.data()), (int64_t)Matcher.size(), 0, out.data(),
                                        (int64_t)out.size(), &n);
  if (!tc.check(ctx, rc, "usv_resolve_match_list")) return;
  for (int64_t k = 0; k < n; ++k) TentativeMatch.push_back({out[k].LeftIndex, out[k].RightIndex, out[k].MatchValue});
}

// P/Main.cpp:483-499 behind the original signature; the join runs on the GPU (usv_resolve.cu). Its output feeds
// MovingObjectDistanceCalculator's index triples; the comma-operator quirk of :492 is kept: (old.RightIndex, 0, 0).
void IDMatcher(std::vector<Match> InterframeMatchIndexes, std::vector<Match> OldInterframeMatchIndexes,
               std::vector<cv::Point3i>& InterframeMatchIndexesComplete) {
  InterframeMatchIndexesComplete.clear();  // :486
  if (InterframeMatchIndexes.empty() || OldInterframeMatchIndexes.empty()) return;
  usv::ThreadContexts& tc = usv::thread_contexts();
  usv_ctx* ctx = tc.get(0);
  if (!ctx) return;
  const usv_match* cur = reinterpret_cast<const usv_match*>(InterframeMatchIndexes.data());
  const usv_match* old = reinterpret_cast<const usv_match*>(OldInterframeMatchIndexes.data());
  const int64_t n_cur = (int64_t)InterframeMatchIndexes.size(), n_old = (int64_t)OldInterframeMatchIndexes.size();
  std::vector<int32_t> out(3 * 64);
  int64_t n = 0;
  int rc = usv_id_matcher(ctx, cur, n_cur, old, n_old, out.data(), (int64_t)out.size() / 3, &n);
  if (rc == USV_OK && n > (int64_t)out.size() / 3) {
    out.resize(3 * (size_t)n);
    rc = usv_id_matcher(ctx, cur, n_cur, old, n_old, out.data(), n, &n);
  }
  if (!tc.check(ctx, rc, "usv_id_matcher")) return;
  for (int64_t k = 0; k < n; ++k) InterframeMatchIndexesComplete.push_back(cv::Point3i(out[3 * k], out[3 * k + 1], out[3 * k + 2]));
}

int RectifyLightingGray(const usv::ImageView& SrcBGR, const short* Map1, const unsigned short* Map2, bool Lighting, unsigned char* Gray,
                        size_t GrayStep, bool OpenCV3Arithmetic, int Device) {
  usv::ThreadContexts& tc = usv::thread_contexts();
  if (!SrcBGR.data || SrcBGR.channels != 3 || !Gray) { tc.last_error = "RectifyLightingGray: needs an 8UC3 frame and an output buffer"; return -1; }
  usv_ctx* ctx = tc.get(Device);
  if (!ctx) return -1;
  usv_preprocess_params p;
  std::memset(&p, 0, sizeof(p));
  p.width = SrcBGR.width; p.height = SrcBGR.height;
  p.src_stride = (int32_t)SrcBGR.step; p.dst_stride = (int32_t)GrayStep;
  p.src_frame_stride = (int64_t)SrcBGR.step * SrcBGR.height; p.dst_frame_stride = (int64_t)GrayStep * SrcBGR.height;
  p.flavour = OpenCV3Arithmetic ? USV_PRE_OPENCV3 : USV_PRE_OPENCV4;
  p.lighting = Lighting ? 1 : 0;
  const int rc = usv_preprocess_host(ctx, SrcBGR.data, 1, Map1, Map2, &p, Gray);
  return tc.check(ctx, rc, "usv_preprocess_host") ? 0 : -1;
}

int BlockSearch(bool CameraSide, const usv::ImageView* ImportGrayThisCamera, const usv::ImageView* ImportGrayOtherCamera,
                const BlockSearchSpec& Spec, std::vector<Match>& ExportMatches, std::vector<double>& ExportDistances) {
  if (!ImportGrayThisCamera || !ImportGrayOtherCamera || !ImportGrayThisCamera->data || !ImportGrayOtherCamera->data ||
      ImportGrayThisCamera->width <= 0 || ImportGrayThisCamera->height <= 0) {
    usv::thread_contexts().last_error = "BlockSearch: empty frame";
    return -1;  // P/Main.cpp:908-911
  }
  BlockSearchSpec s = Spec;
  s.CameraSide = CameraSide;
  ExportMatches.clear();
  ExportDistances.clear();
  usv::ThreadContexts& tc = usv::thread_contexts();
  if (!same_geometry(*ImportGrayThisCamera, *ImportGrayOtherCamera)) { tc.last_error = "BlockSearch: frames of different geometry"; return -1; }
  usv_ctx* ctx = tc.get(s.Device);
  if (!ctx) return -1;
  const usv_search_params p = to_params(s);
  const usv_frame_desc f = to_frame(*ImportGrayThisCamera);
  int32_t nx = 0, ny = 0;
  if (usv_grid_dims(&f, &p, &nx, &ny, nullptr) != USV_OK) { tc.last_error = "BlockSearch: template does not fit the frame"; return -1; }
  const size_t n = (size_t)nx * ny;
  // generate -> resolve -> distance on the device; the survivors land in thread-local buffers and are appended in bulk
  static thread_local std::vector<usv_match> rec;
  static thread_local std::vector<double> dist;
  if (rec.size() < n) { rec.resize(n); dist.resize(n); }
  int64_t n_out = 0;
  const int rc = usv_block_search_host(ctx, ImportGrayThisCamera->data, ImportGrayOtherCamera->data, &f, &p, rec.data(), dist.data(), (int64_t)n, &n_out);
  if (!tc.check(ctx, rc, "usv_block_search_host")) return -1;
  const Match* as_match = reinterpret_cast<const Match*>(rec.data());
  ExportMatches.assign(as_match, as_match + n_out);
  ExportDistances.assign(dist.begin(), dist.begin() + n_out);
  return 0;
}

int BlockSearchPinHostBuffer(void* Buffer, size_t Bytes, int Device) {
  usv::ThreadContexts& tc = usv::thread_contexts();
  usv_ctx* ctx = tc.get(Device);
  if (!ctx) return -1;
  return tc.check(ctx, usv_host_register(ctx, Buffer, Bytes), "usv_host_register") ? 0 : -1;
}

int BlockSearchUnpinHostBuffer(void* Buffer, int Device) {
  usv::ThreadContexts& tc = usv::thread_contexts();
  usv_ctx* ctx = tc.get(Device);
  if (!ctx) return -1;
  return tc.check(ctx, usv_host_unregister(ctx, Buffer), "usv_host_unregister") ? 0 : -1;
}

int DistanceTable(const BlockSearchSpec& Spec, int Count, std::vector<double>& Table) {
  usv::ThreadContexts& tc = usv::thread_contexts();
  usv_ctx* ctx = tc.get(Spec.Device);
  if (!ctx || Count <= 0) return -1;
  Table.assign((size_t)Count, 0.0);
  if (Spec.Distance == BlockSearchSpec::NoDistance) return 0;
  return tc.check(ctx, usv_distance_lut(ctx, (int)Spec.Distance, Count, Table.data()), "usv_distance_lut") ? 0 : -1;
}

namespace {
struct BatchWorker {
  std::mutex busy;
  usv_ctx* ctx = nullptr;
  usv_stream* st = nullptr;
  usv_frame_desc f;
  usv_search_params p;
  uint32_t mask = 0;
  int pps = 0, n_slots = 0;
};
// never destroyed: the CUDA runtime may already be gone when static destructors run
BatchWorker& batch_worker(int device) {
  static std::mutex m;
  static std::map<int, BatchWorker*>* all = new std::map<int, BatchWorker*>();
  std::lock_guard<std::mutex> lock(m);
  BatchWorker*& w = (*all)[device];
  if (!w) w = new BatchWorker();
  return *w;
}
}  // namespace

// One worker per device: context + pinned ring (usv_stream) + one CUDA stream per slot. The worker feeds its contiguous
// block of pairs through the ring, frames straight from the caller's arrays, results straight into its slice of the
// caller's arrays (usv_stream_submit_io): no host-side copy, no shared state between workers, no inter-GPU exchange.
int BlockSearchBatch(const unsigned char* LeftFrames, const unsigned char* RightFrames, int NumPairs, int Width, int Height, size_t Step,
                     size_t FrameStep, const BlockSearchSpec& Spec, const std::vector<int>& Devices, unsigned short* ResolvedDisparity,
                     unsigned short* RawCost, BlockSearchBatchStats* Stats) {
  usv::ThreadContexts& tc0 = usv::thread_contexts();
  if (!LeftFrames || !RightFrames || !ResolvedDisparity || NumPairs < 0 || Devices.empty() || Devices.size() > 16) {
    tc0.last_error = "BlockSearchBatch: bad arguments";
    return -1;
  }
  const usv_search_params p = to_params(Spec);
  usv_frame_desc f;
  f.width = Width; f.height = Height; f.channels = 1;
  f.row_stride = (int32_t)Step; f.frame_stride = (int64_t)FrameStep;
  int32_t nx = 0, ny = 0;
  if (usv_grid_dims(&f, &p, &nx, &ny, nullptr) != USV_OK) { tc0.last_error = "BlockSearchBatch: template does not fit the frame"; return -1; }
  const size_t n_win = (size_t)nx * ny;
  const int G = (int)Devices.size();
  std::vector<std::string> errors(G);
  std::vector<long long> done(G, 0);
  const auto t0 = std::chrono::steady_clock::now();
  auto worker = [&](int g) {
    // pair p -> device floor(p * G / N): contiguous blocks (SURVEY 8e)
    const long long lo = ((long long)g * NumPairs + G - 1) / G, hi = ((long long)(g + 1) * NumPairs + G - 1) / G;
    if (hi <= lo) return;
    // the device's worker state (context, pinned ring, streams) outlives the call: the next batch of the same geometry
    // starts without a single allocation
    BatchWorker& bw = batch_worker(Devices[g]);
    std::lock_guard<std::mutex> lock(bw.busy);
    if (!bw.ctx && usv_create(Devices[g], &bw.ctx) != USV_OK) {
      bw.ctx = nullptr;
      errors[g] = "usv_create failed: no usable sm_100 CUDA device; there is no CPU fallback";
      return;
    }
    usv_ctx* ctx = bw.ctx;
    const int pps = (int)std::min<long long>(32, hi - lo), n_slots = (int)std::min<long long>(6, (hi - lo + pps - 1) / pps);
    const uint32_t mask = USV_OUT_RESOLVED_DISPARITY_U16 | (RawCost ? USV_OUT_RAW_COST_U16 : 0u);
    int rc = USV_OK;
    if (!bw.st || std::memcmp(&bw.f, &f, sizeof(f)) || std::memcmp(&bw.p, &p, sizeof(p)) || bw.mask != mask || bw.pps < pps || bw.n_slots < n_slots) {
      if (bw.st) usv_stream_destroy(bw.st);
      bw.st = nullptr;
      rc = usv_stream_create(ctx, &f, &p, pps, n_slots, mask, &bw.st);
      if (rc != USV_OK) { bw.st = nullptr; errors[g] = std::string("usv_stream_create: ") + usv_last_error(ctx); return; }
      bw.f = f; bw.p = p; bw.mask = mask; bw.pps = pps; bw.n_slots = n_slots;
    }
    usv_stream* st = bw.st;
    long long submitted = lo, waited = lo;
    int slot_sub = 0, slot_wait = 0, in_flight = 0;
    while (waited < hi && rc == USV_OK) {
      if (submitted < hi && in_flight < n_slots) {
        const int cnt = (int)std::min<long long>(pps, hi - submitted);
        usv_outputs dst;
        std::memset(&dst, 0, sizeof(dst));
        dst.resolved_disparity_u16 = ResolvedDisparity + (size_t)submitted * n_win;
        if (RawCost) dst.raw_cost_u16 = RawCost + (size_t)submitted * n_win;
        rc = usv_stream_submit_io(st, slot_sub, LeftFrames + (size_t)submitted * FrameStep, RightFrames + (size_t)submitted * FrameStep, &f,
                                  cnt, &dst);
        submitted += cnt;
        slot_sub = (slot_sub + 1) % n_slots;
        ++in_flight;
      } else {
        rc = usv_stream_wait(st, slot_wait);
        waited = std::min<long long>(hi, waited + pps);
        slot_wait = (slot_wait + 1) % n_slots;
        --in_flight;
      }
    }
    if (rc != USV_OK) errors[g] = std::string("stream: ") + usv_last_error(ctx);
    done[g] = waited - lo;
  };
  std::vector<std::thread> threads;
  for (int g = 1; g < G; ++g) threads.emplace_back(worker, g);
  worker(0);  // the calling thread is the first worker
  for (auto& t : threads) t.join();
  if (Stats) {
    Stats->Seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    Stats->DevicesUsed = G;
    for (int g = 0; g < G; ++g) Stats->PairsPerDevice[g] = done[g];
  }
  for (int g = 0; g < G; ++g)
    if (!errors[g].empty()) { tc0.last_error = "BlockSearchBatch, device " + std::to_string(Devices[g]) + ": " + errors[g]; return -1; }
  tc0.last_error.clear();
  return 0;
}
