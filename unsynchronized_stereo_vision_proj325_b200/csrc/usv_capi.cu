// usv_capi.cu — the C-ABI of include/usv_b200.h: context, validation, kernel
// dispatch, host-buffer paths, the pinned streaming ring and host pairing.
// No CPU compute path exists here: without a CUDA device usv_create fails.
#include <cuda_runtime.h>

#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <algorithm>
#include <cstring>
#include <initializer_list>
#include <memory>
#include <new>
#include <vector>

#include "usv_common.cuh"

namespace usv {
// the direct form; census runs in chunks of pairs whose census frames the scratch holds (at least one pair's)
cudaError_t launch_direct(const DevJob& J, int n_pairs, void* d_scratch, size_t scratch_bytes, cudaStream_t st, int* n_launches);
bool direct_supported(const DevJob& J);
// the dense sweeps, for dense stride-1 jobs of one or three planes: coverage (usv_dense.cu: the SAD sweep, for a batch of
// n_pairs; usv_dense_corr.cu: the correlation sweep that serves the job, Sweep::kNone if none), pair scratch, launch
// (with at least one pair's scratch; launches add to *n_launches)
bool dense_sad_covers(const DevJob& J, int n_pairs);
size_t dense_scratch_bytes_per_pair(const DevJob& J);
cudaError_t launch_dense(const DevJob& J, int n_pairs, void* d_scratch, size_t scratch_bytes, cudaStream_t st, int* n_launches);
Sweep corr_sweep(const DevJob& J);
size_t corr_scratch_bytes_per_pair(const DevJob& J);
cudaError_t launch_dense_corr(const DevJob& J, Sweep sweep, int n_pairs, void* d_scratch, size_t scratch_bytes, cudaStream_t st,
                              int* n_launches);
cudaError_t launch_contour_descriptors(const int* pts, const int* off, int n, double* desc, cudaStream_t st);
cudaError_t launch_contour_costs(const double* dl, int nl, const double* dr, int nr, double* cost, cudaStream_t st);
size_t resolve_workspace_bytes(long long n);
cudaError_t launch_resolve(const usv_match* d_in, long long n, int skip_unmatched, usv_match* d_out, long long cap, long long* d_n_out,
                           void* d_ws, size_t ws_bytes, cudaStream_t st, int* n_launches);
size_t id_matcher_workspace_bytes(long long n_cur);
bool resolve_rows_supported(int nx, int nxc);
struct ResolveRowsSrc {
  const uint16_t* disparity_u16;
  const uint16_t* raw_cost_u16;
  const uint32_t* raw_cost;
  const uint32_t* right_index;
  const usv_match* matches;
};
cudaError_t launch_resolve_rows(const ResolveRowsSrc& S, bool integer_values, int nx, int ny, int sx, int nxc, long long n_templates,
                                int camera_side, int n_pairs, uint16_t* d_out, cudaStream_t st);
cudaError_t launch_id_matcher(const usv_match* d_cur, long long n_cur, const usv_match* d_old, long long n_old, int* d_out3,
                              long long cap, long long* d_n_out, void* d_ws, size_t ws_bytes, cudaStream_t st);
size_t preprocess_scratch_bytes(int width, int height, int n_frames);
cudaError_t launch_preprocess(int device, const uint8_t* d_src, uint8_t* d_dst, const short* d_map1, const uint16_t* d_map2, int n_frames,
                              int width, int height, int src_stride, int dst_stride, long long src_frame_stride,
                              long long dst_frame_stride, int flavour, int lighting, void* d_scratch, cudaStream_t st, int* n_launches);
cudaError_t run_issue_probe(int which, int sms, double target_ms, double* lane_inst_per_s, uint32_t* d_scratch, cudaStream_t st);
cudaError_t launch_disparity_to_distance(const int* d_disp, long long n, int kind, double* d_out, cudaStream_t st);
cudaError_t launch_build_distance_lut(double* d_lut, int n, int kind, cudaStream_t st);
cudaError_t launch_match_list_distance(const usv_match* d_list, const long long* d_n, long long cap, int nx, int sx, int nxc, int camera_side,
                                       int kind, const double* lut, int lut_n, double* d_out, cudaStream_t st);
cudaError_t launch_moving_object_distance(int camera_side, long long t_this, const float* this_xy, int n_this, const float* other_xy,
                                          int n_other, const float* old_xy, int n_old, const float* older_xy, int n_older,
                                          const int* idx3, int n_idx, long long t_other, long long t_old, long long t_older,
                                          double* out, cudaStream_t st);
cudaError_t launch_coordinate_position(int camera_side, const double* dist, const float* xy, long long n, double* xyz, cudaStream_t st);
cudaError_t launch_subpixel_refine(const DevJob& J, int n_pairs, const uint32_t* d_right_index, int* d_x16, double* d_dist,
                                   cudaStream_t st);
}  // namespace usv

namespace usv { int g_sm_count = 148; }

using usv::DevJob;

// Device memory, or pinned host memory when kPinned, that frees itself. Whoever destroys one has set its device and
// synchronised every stream that may still use it.
template <bool kPinned>
struct Buf {
  void* p = nullptr;
  size_t cap = 0;
  Buf() = default;
  Buf(const Buf&) = delete;
  Buf& operator=(const Buf&) = delete;
  Buf(Buf&& o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
  ~Buf() { release(); }
  cudaError_t release() {
    const cudaError_t e = !p ? cudaSuccess : kPinned ? cudaFreeHost(p) : cudaFree(p);
    p = nullptr;
    cap = 0;
    return e;
  }
  // exactly `bytes` into an empty buffer; host_flags are the cudaHostAlloc flags of pinned memory
  cudaError_t alloc(size_t bytes, unsigned host_flags = cudaHostAllocDefault) {
    const cudaError_t e = kPinned ? cudaHostAlloc(&p, bytes, host_flags) : cudaMalloc(&p, bytes);
    if (e == cudaSuccess) cap = bytes;
    else p = nullptr;
    return e;
  }
};
using DevBuf = Buf<false>;
using PinnedBuf = Buf<true>;

static const int kNumOut = 9;
static const size_t kOutElem[kNumOut] = {sizeof(usv_match), 4, 4, 8, 8, 4, 2, 2, 2};

struct usv_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;  // used by the *_host entry points
  char err[512] = {0};
  std::atomic<long long> launches{0};
  const char* last_kernel = "none";
  // distance LUT cache (by kind), [lut_n] doubles. Grow-only: a LUT that is replaced by a longer one stays allocated
  // until usv_destroy (kernels in flight on other streams of this context may still read it)
  DevBuf lut[3];
  int lut_n[3] = {0, 0, 0};
  std::vector<DevBuf> retired;
  // status word the kernels can raise (mapped pinned host memory: readable by the host without a copy)
  PinnedBuf status;
  int* d_status = nullptr;
  int corr_kernel = USV_CORR_KERNEL_AUTO;
  std::atomic<int> open_streams{0};  // usv_destroy refuses while a usv_stream of this context is alive
  // grow-only pinned staging of usv_block_search_host (frames in, match list + distances out)
  PinnedBuf pin[3];
  // grow-only scratch for the host paths
  DevBuf in_l, in_r, tx, ty, rows_u32, rows_f64, out[kNumOut], misc[8], resolve_ws, pre_ws, corr_ws, win_ws;
  DevBuf sub_ri, sub_x16, sub_dist;  // usv_match_dense_subpixel_host: winners' RightIndex, refined disparity, distance
  ~usv_ctx() { if (stream) cudaStreamDestroy(stream); }
};

static int fail(usv_ctx* c, int code, const char* fmt, ...) {
  if (c) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(c->err, sizeof(c->err), fmt, ap);
    va_end(ap);
  }
  return code;
}
#define CU(call)                                                                                         \
  do {                                                                                                   \
    cudaError_t e_ = (call);                                                                             \
    if (e_ != cudaSuccess) return fail(ctx, USV_ERR_CUDA, "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

template <bool kPinned>
static int grow(usv_ctx* ctx, Buf<kPinned>& b, size_t bytes) {
  if (bytes <= b.cap) return USV_OK;
  CU(b.release());
  const size_t want = bytes + bytes / 4 + (kPinned ? 4096 : 256);
  const cudaError_t e = b.alloc(want);
  if (e != cudaSuccess)
    return fail(ctx, USV_ERR_NOMEM, "%s(%zu): %s", kPinned ? "cudaHostAlloc" : "cudaMalloc", want, cudaGetErrorString(e));
  return USV_OK;
}

// pair scratch of a dense sweep: room for every pair up to this cap (at least one pair); the sweeps run the pairs in
// chunks of what it holds
static const size_t kPairScratchCap = (size_t)3 << 29;  // 1.5 GB

static int grow_pair_scratch(usv_ctx* ctx, DevBuf& ws, size_t per_pair, int32_t n_pairs) {
  size_t want = per_pair * (size_t)n_pairs;
  if (want > kPairScratchCap) want = std::max(per_pair, kPairScratchCap / per_pair * per_pair);
  return grow(ctx, ws, want);
}

// every array of `arrs` that is null (not asked for by the caller) is pointed at its share of scratch `ws`
struct ArrayOrScratch {
  void** arr;
  size_t bytes;
};
static int or_scratch(usv_ctx* ctx, DevBuf& ws, std::initializer_list<ArrayOrScratch> arrs) {
  size_t total = 0;
  for (const ArrayOrScratch& a : arrs) total += *a.arr ? 0 : a.bytes;
  const int rc = grow(ctx, ws, total);
  if (rc) return rc;
  uint8_t* q = (uint8_t*)ws.p;
  for (const ArrayOrScratch& a : arrs)
    if (!*a.arr) { *a.arr = q; q += a.bytes; }
  return USV_OK;
}

// device layout of host frames: rows at a 128-byte pitch, frames packed
static usv_frame_desc device_frame_desc(const usv_frame_desc* f) {
  usv_frame_desc d = *f;
  d.row_stride = (f->width * f->channels + 127) & ~127;
  d.frame_stride = (int64_t)d.row_stride * f->height;
  return d;
}

// H2D of `n` consecutive host frames (layout `hf`) into consecutive device frames (layout `df`) from `dst` on: one copy
// when the layouts agree, one 2D copy when the host frames are packed, one 2D copy per frame otherwise
static int copy_frames(usv_ctx* ctx, uint8_t* dst, const usv_frame_desc& df, const uint8_t* src, const usv_frame_desc* hf, int32_t n,
                       cudaStream_t st) {
  const int row_bytes = hf->width * hf->channels;
  const bool packed = n == 1 || hf->frame_stride == (int64_t)hf->row_stride * hf->height;
  if (packed && hf->row_stride == df.row_stride) {
    CU(cudaMemcpyAsync(dst, src, (size_t)df.frame_stride * n, cudaMemcpyHostToDevice, st));
  } else if (packed) {
    CU(cudaMemcpy2DAsync(dst, df.row_stride, src, hf->row_stride, row_bytes, (size_t)hf->height * n, cudaMemcpyHostToDevice, st));
  } else {
    for (int i = 0; i < n; ++i)
      CU(cudaMemcpy2DAsync(dst + (size_t)i * df.frame_stride, df.row_stride, src + (size_t)i * hf->frame_stride, hf->row_stride,
                           row_bytes, hf->height, cudaMemcpyHostToDevice, st));
  }
  return USV_OK;
}

static void** out_slot(usv_outputs* o, int i) {
  switch (i) {
    case 0: return (void**)&o->matches;
    case 1: return (void**)&o->right_index;
    case 2: return (void**)&o->raw_cost;
    case 3: return (void**)&o->score;
    case 4: return (void**)&o->distance;
    case 5: return (void**)&o->distance_f32;
    case 6: return (void**)&o->disparity_u16;
    case 7: return (void**)&o->raw_cost_u16;
    default: return (void**)&o->resolved_disparity_u16;
  }
}

// ---- validation + job construction ---------------------------------------------
static int check_common(usv_ctx* ctx, const usv_frame_desc* f, const usv_search_params* p, int32_t n_pairs) {
  if (!ctx) return USV_ERR_INVALID_ARG;
  if (!f || !p) return fail(ctx, USV_ERR_INVALID_ARG, "null frame/params");
  if (n_pairs < 0 || n_pairs > 65535) return fail(ctx, USV_ERR_INVALID_ARG, "n_pairs %d out of [0, 65535]", n_pairs);
  if (f->width <= 0 || f->height <= 0 || f->channels < 1 || f->channels > 4)
    return fail(ctx, USV_ERR_INVALID_ARG, "bad frame %dx%dx%d", f->width, f->height, f->channels);
  if (f->row_stride < f->width * f->channels) return fail(ctx, USV_ERR_INVALID_ARG, "row_stride %d < width*channels", f->row_stride);
  if (n_pairs > 1 && f->frame_stride < (int64_t)f->row_stride * f->height)
    return fail(ctx, USV_ERR_INVALID_ARG, "frame_stride smaller than one frame");
  if (p->tmpl_w <= 0 || p->tmpl_h <= 0 || p->tmpl_w > f->width || p->tmpl_h > f->height)
    return fail(ctx, USV_ERR_INVALID_ARG, "template %dx%d does not fit frame %dx%d", p->tmpl_w, p->tmpl_h, f->width, f->height);
  if ((int64_t)p->tmpl_w * p->tmpl_h * f->channels > 32768)
    return fail(ctx, USV_ERR_UNSUPPORTED, "template of %lld bytes exceeds 32768 (u32 cost accumulators)",
                (long long)p->tmpl_w * p->tmpl_h * f->channels);
  if (p->tmpl_w * f->channels > 1024) return fail(ctx, USV_ERR_UNSUPPORTED, "template row wider than 1024 bytes");
  if (p->stride_x <= 0 || p->stride_y <= 0) return fail(ctx, USV_ERR_INVALID_ARG, "stride must be positive");
  if (p->search_min > p->search_max) return fail(ctx, USV_ERR_INVALID_ARG, "search_min > search_max");
  if (p->search_min < -(1 << 24) || p->search_max > (1 << 24)) return fail(ctx, USV_ERR_INVALID_ARG, "search range beyond +-2^24");
  if (p->cost_kind < USV_COST_SAD || p->cost_kind > USV_COST_CENSUS) return fail(ctx, USV_ERR_INVALID_ARG, "unknown cost_kind %d", p->cost_kind);
  if (p->distance_kind < USV_DIST_NONE || p->distance_kind > USV_DIST_POWERLAW)
    return fail(ctx, USV_ERR_INVALID_ARG, "unknown distance_kind %d", p->distance_kind);
  if (p->camera_side != USV_LEFT_CAM && p->camera_side != USV_RIGHT_CAM) return fail(ctx, USV_ERR_INVALID_ARG, "camera_side must be 0 or 1");
  return USV_OK;
}

// raw_cost_u16 is lossless or refused: every SAD or census cost of the template must fit 16 bits below 0xFFFF, the
// "no candidate" value
static int check_cost_u16(usv_ctx* ctx, const usv_frame_desc* f, const usv_search_params* p) {
  const long long unit = p->cost_kind == USV_COST_SAD ? 255 : p->cost_kind == USV_COST_CENSUS ? 8 : 0;
  if (unit == 0 || unit * p->tmpl_w * p->tmpl_h * f->channels >= 0xFFFFll)
    return fail(ctx, USV_ERR_UNSUPPORTED, "raw_cost_u16 needs SAD with 255*tmpl_w*tmpl_h*channels < 65535 or CENSUS with 8*... < 65535");
  return USV_OK;
}

// only the direct form serves sparse lists and whatever the dense sweeps do not cover; some narrow, tall templates do not
// fit its shared memory
static int check_direct(usv_ctx* ctx, const DevJob& J) {
  if (!usv::direct_supported(J))
    return fail(ctx, USV_ERR_UNSUPPORTED, "template %dx%dx%d: no kernel serves this shape (direct form: shared memory)", J.tw, J.th,
                J.channels);
  return USV_OK;
}

// a kernel gave up (today: a tcgen05 completion wait beyond its wall-clock bound): report it once, as an error
static int check_dev_status(usv_ctx* ctx) {
  volatile int* h_status = (volatile int*)ctx->status.p;
  if (h_status && *h_status != 0) {
    const int s = *h_status;
    *h_status = 0;
    return fail(ctx, USV_ERR_CUDA, "device status %d: a kernel abandoned a wait (results of the affected call are invalid)", s);
  }
  return USV_OK;
}

static void fill_job(usv_ctx* ctx, DevJob& J, const uint8_t* l, const uint8_t* r, const usv_frame_desc* f, const usv_search_params* p,
                     const usv_outputs* o) {
  memset(&J, 0, sizeof(J));
  J.status = ctx->d_status;
  J.corr_kernel = ctx->corr_kernel;
  J.left = l; J.right = r;
  J.frame_stride = f->frame_stride;
  J.width = f->width; J.height = f->height; J.channels = f->channels; J.row_stride = f->row_stride;
  J.tw = p->tmpl_w; J.th = p->tmpl_h; J.dmin = p->search_min; J.dmax = p->search_max;
  J.sx = p->stride_x; J.sy = p->stride_y;
  J.cost_kind = p->cost_kind; J.camera_side = p->camera_side; J.distance_kind = p->distance_kind;
  J.nxc = f->width - p->tmpl_w + 1; J.nyc = f->height - p->tmpl_h + 1;
  J.nx = (J.nxc - 1) / p->stride_x + 1; J.ny = (J.nyc - 1) / p->stride_y + 1;
  J.row_bytes = p->tmpl_w * f->channels;
  J.n_elems = p->tmpl_w * p->tmpl_h * f->channels;
  J.accept_threshold = p->accept_threshold;
  J.n_templates = J.nx * J.ny;
  if (o) J.out = *o;
}

static int ensure_lut(usv_ctx* ctx, int kind, int width, cudaStream_t st, const double** lut) {
  *lut = nullptr;
  if (kind == USV_DIST_NONE) return USV_OK;
  if (ctx->lut_n[kind] < width) {
    // (re)build on the device with the same device function the kernels use
    if (ctx->lut[kind].p) { ctx->retired.push_back(std::move(ctx->lut[kind])); ctx->lut_n[kind] = 0; }
    int n = width < 4096 ? 4096 : width;
    CU(ctx->lut[kind].alloc(sizeof(double) * n));
    CU(usv::launch_build_distance_lut((double*)ctx->lut[kind].p, n, kind, st));
    CU(cudaStreamSynchronize(st));  // one-time; other streams of this context may read it next
    ctx->launches++;
    ctx->lut_n[kind] = n;
  }
  *lut = (const double*)ctx->lut[kind].p;
  return USV_OK;
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// ---- lifetime ---------------------------------------------------------------------
extern "C" int usv_abi_version(void) { return USV_ABI_VERSION; }

extern "C" int usv_create(int device, usv_ctx** out) {
  if (!out) return USV_ERR_INVALID_ARG;
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0) return USV_ERR_NO_DEVICE;  // no CPU fallback: fail loudly
  if (device < 0 || device >= n) return USV_ERR_INVALID_ARG;
  if (cudaSetDevice(device) != cudaSuccess) return USV_ERR_CUDA;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return USV_ERR_CUDA;
  // the library holds sm_100a cubins only (arch-specific, not forward compatible): any other part would fail every
  // launch with "no kernel image", so it is refused here
  if (prop.major != 10 || prop.minor != 0) return USV_ERR_NO_DEVICE;
  usv_ctx* c = new (std::nothrow) usv_ctx();
  if (!c) return USV_ERR_NOMEM;
  c->device = device;
  usv::g_sm_count = prop.multiProcessorCount;
  if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess ||
      c->status.alloc(sizeof(int), cudaHostAllocMapped) != cudaSuccess ||
      cudaHostGetDevicePointer((void**)&c->d_status, c->status.p, 0) != cudaSuccess) {
    delete c;
    return USV_ERR_CUDA;
  }
  *(int*)c->status.p = 0;
  *out = c;
  return USV_OK;
}

extern "C" int usv_destroy(usv_ctx* ctx) {
  if (!ctx) return USV_ERR_INVALID_ARG;
  if (ctx->open_streams.load() > 0)
    return fail(ctx, USV_ERR_INVALID_ARG, "%d usv_stream(s) of this context are still open: destroy them first", ctx->open_streams.load());
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  delete ctx;
  return USV_OK;
}

extern "C" const char* usv_last_error(const usv_ctx* ctx) { return ctx ? ctx->err : "null context"; }
extern "C" int64_t usv_launch_count(const usv_ctx* ctx) { return ctx ? (int64_t)ctx->launches.load() : -1; }
extern "C" const char* usv_last_kernel(const usv_ctx* ctx) { return ctx ? ctx->last_kernel : "none"; }
extern "C" int usv_set_option(usv_ctx* ctx, int32_t key, int64_t value) {
  if (!ctx) return USV_ERR_INVALID_ARG;
  if (key == USV_OPT_CORR_KERNEL) {
    if (value < USV_CORR_KERNEL_AUTO || value > USV_CORR_KERNEL_TCGEN05) return fail(ctx, USV_ERR_INVALID_ARG, "USV_OPT_CORR_KERNEL: value %lld", (long long)value);
    ctx->corr_kernel = (int)value;
    return USV_OK;
  }
  return fail(ctx, USV_ERR_INVALID_ARG, "unknown option %d", key);
}
extern "C" int usv_device_status(usv_ctx* ctx) { return ctx ? check_dev_status(ctx) : USV_ERR_INVALID_ARG; }

extern "C" int usv_grid_dims(const usv_frame_desc* f, const usv_search_params* p, int32_t* nx, int32_t* ny, int64_t* cand_evals) {
  if (!f || !p) return USV_ERR_INVALID_ARG;
  int nxc = f->width - p->tmpl_w + 1, nyc = f->height - p->tmpl_h + 1;
  if (nxc <= 0 || nyc <= 0 || p->stride_x <= 0 || p->stride_y <= 0) return USV_ERR_INVALID_ARG;
  int gx = (nxc - 1) / p->stride_x + 1, gy = (nyc - 1) / p->stride_y + 1;
  int64_t per_row = 0;
  for (int ix = 0; ix < gx; ++ix) {
    int lo, hi;
    usv::cand_range(ix * p->stride_x, nxc, p->camera_side, p->search_min, p->search_max, &lo, &hi);
    if (hi >= lo) per_row += hi - lo + 1;
  }
  if (nx) *nx = gx;
  if (ny) *ny = gy;
  if (cand_evals) *cand_evals = per_row * gy;
  return USV_OK;
}

static int resolve_device(usv_ctx* ctx, const usv_match* d_in, int64_t n, int32_t skip_unmatched, usv_match* d_out, int64_t cap,
                          int64_t* d_n_out, cudaStream_t st);

// ---- matching: device pointers -----------------------------------------------------
// The sweep that serves a matching call of n_pairs and the pair scratch it needs per pair, chosen before anything is
// allocated or launched, in the order of the dispatch table of DESIGN §4
struct MatchPlan {
  usv::Sweep sweep;
  size_t scratch_per_pair;
};
static MatchPlan plan_match(const DevJob& J, int n_pairs) {
  using usv::Sweep;
  const bool dense = !J.tx && J.sx == 1 && J.sy == 1 && (J.channels == 1 || J.channels == 3);
  // USV_CORR_KERNEL_ALU also moves colour SAD to the ALU correlation kernel (a test / measurement aid); census stays
  const bool colour_sad_on_alu = J.cost_kind == USV_COST_SAD && J.channels == 3 && J.corr_kernel == USV_CORR_KERNEL_ALU;
  if (dense && !colour_sad_on_alu && usv::dense_sad_covers(J, n_pairs))
    return {J.cost_kind == USV_COST_CENSUS ? Sweep::kCensus : Sweep::kSad, usv::dense_scratch_bytes_per_pair(J)};
  const Sweep corr = dense ? usv::corr_sweep(J) : Sweep::kNone;
  return corr != Sweep::kNone ? MatchPlan{corr, usv::corr_scratch_bytes_per_pair(J)}
                              : MatchPlan{Sweep::kDirect, usv::census_scratch_bytes_per_pair(J)};
}
// by usv::Sweep: the kernel usv_last_kernel reports, and what a failed launch of it is called
static const char* const kSweepKernel[] = {"dense_sad_argmin_kernel", "dense_census_argmin_kernel", "dense_corr_argmin_kernel",
                                           "dense_corr_mma_kernel", "dense_corr_umma_kernel", "block_cost_argmin_direct"};
static const char* const kSweepLaunch[] = {"dense", "dense census", "dense correlation", "dense correlation", "dense correlation", "direct"};

// the matching kernels of one call
static int dispatch_match(usv_ctx* ctx, const DevJob& J, int32_t n_pairs, cudaStream_t st, DevBuf* corr_ws) {
  const MatchPlan plan = plan_match(J, n_pairs);
  int rc, nl = 0;
  if (plan.sweep == usv::Sweep::kDirect && (rc = check_direct(ctx, J))) return rc;
  // the scratch (census frames, colour planes of the SAD sweep, planes + window statistics of the correlation sweeps)
  // belongs to whoever owns the stream: launches on different streams must not share it. Jobs that need none (the direct
  // form of the costs other than census, gray SAD) grow nothing.
  DevBuf& ws = corr_ws ? *corr_ws : ctx->corr_ws;
  if ((rc = grow_pair_scratch(ctx, ws, plan.scratch_per_pair, n_pairs))) return rc;
  const cudaError_t e = plan.sweep == usv::Sweep::kDirect ? usv::launch_direct(J, n_pairs, ws.p, ws.cap, st, &nl)
                        : plan.sweep == usv::Sweep::kSad || plan.sweep == usv::Sweep::kCensus
                            ? usv::launch_dense(J, n_pairs, ws.p, ws.cap, st, &nl)
                            : usv::launch_dense_corr(J, plan.sweep, n_pairs, ws.p, ws.cap, st, &nl);
  if (e != cudaSuccess) return fail(ctx, USV_ERR_CUDA, "%s launch: %s", kSweepLaunch[(int)plan.sweep], cudaGetErrorString(e));
  ctx->launches += nl;
  ctx->last_kernel = kSweepKernel[(int)plan.sweep];
  return USV_OK;
}

// the arrays the resolved disparity map reads the winners from
enum WinnerSrc { kWinDisparity, kWinRightIndex, kWinMatches };

static WinnerSrc winner_src(const usv_search_params* p, const usv_outputs& o) {
  if (p->cost_kind == USV_COST_NCC || p->cost_kind == USV_COST_ZNCC) return kWinMatches;  // the value of a correlation winner is an f64 score
  // a u16 disparity names x' only when no candidate lies on the other side of the window (search_min >= 0): negative
  // disparities are stored modulo 2^16 and -1 would read as USV_NO_DISPARITY; such ranges resolve from RightIndex
  const bool disp_ok = p->search_min >= 0;
  if (disp_ok && o.disparity_u16 && (o.raw_cost_u16 || o.raw_cost)) return kWinDisparity;
  if (o.right_index && o.raw_cost) return kWinRightIndex;
  return disp_ok ? kWinDisparity : kWinRightIndex;
}

static int match_device(usv_ctx* ctx, const uint8_t* d_left, const uint8_t* d_right, const usv_frame_desc* f, int32_t n_pairs,
                        const usv_search_params* p, const usv_outputs* d_out, const int32_t* d_tx, const int32_t* d_ty,
                        int32_t n_templates, uint32_t* d_cost_rows, double* d_score_rows, int32_t row_cap, cudaStream_t st, DevBuf* corr_ws = nullptr,
                        DevBuf* win_ws = nullptr) {
  int rc = check_common(ctx, f, p, n_pairs);
  if (rc) return rc;
  if (!d_left || !d_right || !d_out) return fail(ctx, USV_ERR_INVALID_ARG, "null device pointer");
  if (!aligned16(d_left) || !aligned16(d_right) || (f->row_stride & 15) || (f->frame_stride & 15))
    return fail(ctx, USV_ERR_INVALID_ARG, "device frames need 16-byte aligned base, row_stride and frame_stride");
  if (d_out->raw_cost_u16 && (rc = check_cost_u16(ctx, f, p))) return rc;
  if (n_pairs == 0) return USV_OK;
  CU(cudaSetDevice(ctx->device));
  DevJob J;
  fill_job(ctx, J, d_left, d_right, f, p, d_out);
  const bool sparse = d_tx != nullptr;
  if (sparse) {
    if (!d_ty || n_templates < 0) return fail(ctx, USV_ERR_INVALID_ARG, "bad template list");
    if (n_templates == 0) return USV_OK;
    J.tx = d_tx; J.ty = d_ty; J.n_templates = n_templates;
    J.cost_rows = d_cost_rows; J.score_rows = d_score_rows; J.row_cap = row_cap;
    if ((d_cost_rows || d_score_rows) && row_cap <= 0) return fail(ctx, USV_ERR_INVALID_ARG, "row_cap must be positive");
  }
  if (J.out.distance || J.out.distance_f32) {
    rc = ensure_lut(ctx, p->distance_kind, f->width, st, &J.dist_lut);
    if (rc) return rc;
  }
  // resolved disparity map: ResolveMatchList over the winners on the device (usv_resolve_rows.cu). It reads the
  // winners from `src`: the caller's arrays when they were asked for, scratch otherwise.
  const bool want_resolved = d_out->resolved_disparity_u16 != nullptr;
  const WinnerSrc src = winner_src(p, J.out);
  if (want_resolved) {
    if (sparse) return fail(ctx, USV_ERR_UNSUPPORTED, "resolved_disparity_u16 is an output of the dense sweep");
    if (!usv::resolve_rows_supported(J.nx, J.nxc)) return fail(ctx, USV_ERR_UNSUPPORTED, "resolved_disparity_u16: rows wider than 2048 windows");
    const size_t n_res = (size_t)J.n_templates * n_pairs;
    DevBuf& ws = win_ws ? *win_ws : ctx->win_ws;
    usv_outputs& o = J.out;
    if (src == kWinDisparity)  // either cost array serves; raw_cost is added when the caller asked for neither
      rc = or_scratch(ctx, ws, {{o.raw_cost_u16 ? (void**)&o.raw_cost_u16 : (void**)&o.raw_cost, 4 * n_res},
                                {(void**)&o.disparity_u16, 2 * n_res}});
    else if (src == kWinRightIndex)
      rc = or_scratch(ctx, ws, {{(void**)&o.raw_cost, 4 * n_res}, {(void**)&o.right_index, 4 * n_res}});
    else
      rc = or_scratch(ctx, ws, {{(void**)&o.matches, sizeof(usv_match) * n_res}});
    if (rc) return rc;
  }
  if ((rc = dispatch_match(ctx, J, n_pairs, st, corr_ws))) return rc;
  if (want_resolved) {
    usv::ResolveRowsSrc S;
    memset(&S, 0, sizeof(S));
    if (src == kWinDisparity) {
      S.disparity_u16 = J.out.disparity_u16; S.raw_cost_u16 = J.out.raw_cost_u16; S.raw_cost = J.out.raw_cost;
    } else if (src == kWinRightIndex) {
      S.right_index = J.out.right_index; S.raw_cost = J.out.raw_cost;
    } else {
      S.matches = J.out.matches;
    }
    cudaError_t e = usv::launch_resolve_rows(S, src != kWinMatches, J.nx, J.ny, J.sx, J.nxc, J.n_templates, J.camera_side, n_pairs,
                                             d_out->resolved_disparity_u16, st);
    if (e != cudaSuccess) return fail(ctx, USV_ERR_CUDA, "resolve rows launch: %s", cudaGetErrorString(e));
    ctx->launches++;
  }
  return USV_OK;
}

extern "C" int usv_match_dense_device(usv_ctx* ctx, const uint8_t* d_left, const uint8_t* d_right, const usv_frame_desc* frame,
                                      int32_t n_pairs, const usv_search_params* params, const usv_outputs* d_out, void* cuda_stream) {
  if (!ctx) return USV_ERR_INVALID_ARG;
  return match_device(ctx, d_left, d_right, frame, n_pairs, params, d_out, nullptr, nullptr, 0, nullptr, nullptr, 0,
                      (cudaStream_t)cuda_stream);
}

extern "C" int usv_match_templates_device(usv_ctx* ctx, const uint8_t* d_left, const uint8_t* d_right, const usv_frame_desc* frame,
                                          int32_t n_pairs, const int32_t* d_tx, const int32_t* d_ty, int32_t n_templates,
                                          const usv_search_params* params, const usv_outputs* d_out, uint32_t* d_cost_rows,
                                          double* d_score_rows, int32_t row_cap, void* cuda_stream) {
  if (!ctx) return USV_ERR_INVALID_ARG;
  if (!d_tx) return fail(ctx, USV_ERR_INVALID_ARG, "null template list");
  return match_device(ctx, d_left, d_right, frame, n_pairs, params, d_out, d_tx, d_ty, n_templates, d_cost_rows, d_score_rows,
                      row_cap, (cudaStream_t)cuda_stream);
}

// ---- sub-pixel refinement of dense winners (usv_subpixel.cu) --------------------------
static int check_subpixel(usv_ctx* ctx, const usv_frame_desc* f, const usv_search_params* p, const void* x16, const void* dist) {
  if (!x16 && !dist) return fail(ctx, USV_ERR_INVALID_ARG, "sub-pixel refinement: both output pointers are NULL");
  // the refinement scores the winner's neighbours from frame bytes; census would need the census frames
  if (p->cost_kind == USV_COST_CENSUS) return fail(ctx, USV_ERR_UNSUPPORTED, "sub-pixel refinement: not available for USV_COST_CENSUS");
  // 16 * d must fit int32
  if (f->width > (1 << 26)) return fail(ctx, USV_ERR_UNSUPPORTED, "sub-pixel refinement: frame wider than 2^26 pixels");
  return USV_OK;
}

static int refine_device(usv_ctx* ctx, const uint8_t* d_left, const uint8_t* d_right, const usv_frame_desc* f, int32_t n_pairs,
                         const usv_search_params* p, const uint32_t* d_ri, int32_t* d_x16, double* d_dist, cudaStream_t st) {
  int rc = check_common(ctx, f, p, n_pairs);
  if (rc || (rc = check_subpixel(ctx, f, p, d_x16, d_dist))) return rc;
  if (!d_left || !d_right || !d_ri) return fail(ctx, USV_ERR_INVALID_ARG, "null device pointer");
  if (!aligned16(d_left) || !aligned16(d_right) || (f->row_stride & 15) || (f->frame_stride & 15))
    return fail(ctx, USV_ERR_INVALID_ARG, "device frames need 16-byte aligned base, row_stride and frame_stride");
  if (n_pairs == 0) return USV_OK;
  CU(cudaSetDevice(ctx->device));
  DevJob J;
  fill_job(ctx, J, d_left, d_right, f, p, nullptr);
  cudaError_t e = usv::launch_subpixel_refine(J, n_pairs, d_ri, d_x16, d_dist, st);
  if (e != cudaSuccess) return fail(ctx, USV_ERR_CUDA, "sub-pixel launch: %s", cudaGetErrorString(e));
  ctx->launches++;
  return USV_OK;
}

extern "C" int usv_refine_subpixel_device(usv_ctx* ctx, const uint8_t* d_left, const uint8_t* d_right, const usv_frame_desc* frame,
                                          int32_t n_pairs, const usv_search_params* params, const uint32_t* d_right_index,
                                          int32_t* d_disparity_x16, double* d_distance, void* cuda_stream) {
  if (!ctx) return USV_ERR_INVALID_ARG;
  return refine_device(ctx, d_left, d_right, frame, n_pairs, params, d_right_index, d_disparity_x16, d_distance,
                       (cudaStream_t)cuda_stream);
}

// ---- matching: host pointers (H2D + kernels + D2H + sync inside) --------------------
// optional step after the dense sweep of match_host: refine its winners into these host arrays (either may be NULL)
struct SubpixelOut {
  int32_t* disparity_x16;
  double* distance;
};

static int match_host(usv_ctx* ctx, const uint8_t* h_left, const uint8_t* h_right, const usv_frame_desc* f, int32_t n_pairs,
                      const usv_search_params* p, const usv_outputs* h_out, const int32_t* h_tx, const int32_t* h_ty,
                      int32_t n_templates, uint32_t* h_cost_rows, double* h_score_rows, int32_t row_cap,
                      const SubpixelOut* sub = nullptr) {
  int rc = check_common(ctx, f, p, n_pairs);
  if (rc) return rc;
  if (!h_left || !h_right || !h_out) return fail(ctx, USV_ERR_INVALID_ARG, "null host pointer");
  if (sub && (rc = check_subpixel(ctx, f, p, sub->disparity_x16, sub->distance))) return rc;
  if (n_pairs == 0) return USV_OK;
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const bool sparse = h_tx != nullptr;
  int64_t n_win;
  if (sparse) {
    if (!h_ty || n_templates < 0) return fail(ctx, USV_ERR_INVALID_ARG, "bad template list");
    const int nxc = f->width - p->tmpl_w + 1, nyc = f->height - p->tmpl_h + 1;
    for (int i = 0; i < n_templates; ++i)
      if (h_tx[i] < 0 || h_tx[i] >= nxc || h_ty[i] < 0 || h_ty[i] >= nyc)
        return fail(ctx, USV_ERR_INVALID_ARG, "template %d at (%d,%d) outside the frame", i, h_tx[i], h_ty[i]);
    n_win = n_templates;
    if (n_templates == 0) return USV_OK;
    DevJob J;
    fill_job(ctx, J, nullptr, nullptr, f, p, nullptr);
    if ((rc = check_direct(ctx, J))) return rc;
  } else {
    int32_t nx, ny;
    if (usv_grid_dims(f, p, &nx, &ny, nullptr)) return fail(ctx, USV_ERR_INVALID_ARG, "bad geometry");
    n_win = (int64_t)nx * ny;
  }
  const int64_t n_res = n_win * n_pairs;
  const usv_frame_desc df = device_frame_desc(f);
  const size_t fbytes = (size_t)df.frame_stride * n_pairs;
  if ((rc = grow(ctx, ctx->in_l, fbytes)) || (rc = copy_frames(ctx, (uint8_t*)ctx->in_l.p, df, h_left, f, n_pairs, st))) return rc;
  if ((rc = grow(ctx, ctx->in_r, fbytes)) || (rc = copy_frames(ctx, (uint8_t*)ctx->in_r.p, df, h_right, f, n_pairs, st))) return rc;
  usv_outputs d_out;
  memset(&d_out, 0, sizeof(d_out));
  usv_outputs ho = *h_out;
  for (int i = 0; i < kNumOut; ++i) {
    if (*out_slot(&ho, i)) {
      if ((rc = grow(ctx, ctx->out[i], kOutElem[i] * n_res))) return rc;
      *out_slot(&d_out, i) = ctx->out[i].p;
    }
  }
  int32_t *d_tx = nullptr, *d_ty = nullptr;
  uint32_t* d_rows = nullptr;
  double* d_srows = nullptr;
  if (sparse) {
    if ((rc = grow(ctx, ctx->tx, sizeof(int32_t) * n_templates))) return rc;
    if ((rc = grow(ctx, ctx->ty, sizeof(int32_t) * n_templates))) return rc;
    d_tx = (int32_t*)ctx->tx.p; d_ty = (int32_t*)ctx->ty.p;
    CU(cudaMemcpyAsync(d_tx, h_tx, sizeof(int32_t) * n_templates, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_ty, h_ty, sizeof(int32_t) * n_templates, cudaMemcpyHostToDevice, st));
    if (h_cost_rows) {
      if ((rc = grow(ctx, ctx->rows_u32, sizeof(uint32_t) * n_res * row_cap))) return rc;
      d_rows = (uint32_t*)ctx->rows_u32.p;
      CU(cudaMemcpyAsync(d_rows, h_cost_rows, sizeof(uint32_t) * n_res * row_cap, cudaMemcpyHostToDevice, st));
    }
    if (h_score_rows) {
      if ((rc = grow(ctx, ctx->rows_f64, sizeof(double) * n_res * row_cap))) return rc;
      d_srows = (double*)ctx->rows_f64.p;
      CU(cudaMemcpyAsync(d_srows, h_score_rows, sizeof(double) * n_res * row_cap, cudaMemcpyHostToDevice, st));
    }
  }
  // the refinement reads the winners' RightIndex: the caller's array when it was asked for, scratch otherwise
  if (sub && (rc = or_scratch(ctx, ctx->sub_ri, {{(void**)&d_out.right_index, 4 * (size_t)n_res}}))) return rc;
  rc = match_device(ctx, (const uint8_t*)ctx->in_l.p, (const uint8_t*)ctx->in_r.p, &df, n_pairs, p, &d_out, d_tx, d_ty, n_templates,
                    d_rows, d_srows, row_cap, st);
  if (rc) return rc;
  if (sub) {
    int32_t* d_x16 = nullptr;
    double* d_dist = nullptr;
    if (sub->disparity_x16) {
      if ((rc = grow(ctx, ctx->sub_x16, 4 * n_res))) return rc;
      d_x16 = (int32_t*)ctx->sub_x16.p;
    }
    if (sub->distance) {
      if ((rc = grow(ctx, ctx->sub_dist, 8 * n_res))) return rc;
      d_dist = (double*)ctx->sub_dist.p;
    }
    if ((rc = refine_device(ctx, (const uint8_t*)ctx->in_l.p, (const uint8_t*)ctx->in_r.p, &df, n_pairs, p, d_out.right_index, d_x16,
                            d_dist, st)))
      return rc;
    if (d_x16) CU(cudaMemcpyAsync(sub->disparity_x16, d_x16, 4 * n_res, cudaMemcpyDeviceToHost, st));
    if (d_dist) CU(cudaMemcpyAsync(sub->distance, d_dist, 8 * n_res, cudaMemcpyDeviceToHost, st));
  }
  for (int i = 0; i < kNumOut; ++i)
    if (*out_slot(&ho, i)) CU(cudaMemcpyAsync(*out_slot(&ho, i), ctx->out[i].p, kOutElem[i] * n_res, cudaMemcpyDeviceToHost, st));
  if (d_rows) CU(cudaMemcpyAsync(h_cost_rows, d_rows, sizeof(uint32_t) * n_res * row_cap, cudaMemcpyDeviceToHost, st));
  if (d_srows) CU(cudaMemcpyAsync(h_score_rows, d_srows, sizeof(double) * n_res * row_cap, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return check_dev_status(ctx);
}

extern "C" int usv_match_dense_host(usv_ctx* ctx, const uint8_t* h_left, const uint8_t* h_right, const usv_frame_desc* frame,
                                    int32_t n_pairs, const usv_search_params* params, const usv_outputs* h_out) {
  if (!ctx) return USV_ERR_INVALID_ARG;
  return match_host(ctx, h_left, h_right, frame, n_pairs, params, h_out, nullptr, nullptr, 0, nullptr, nullptr, 0);
}

extern "C" int usv_match_templates_host(usv_ctx* ctx, const uint8_t* h_left, const uint8_t* h_right, const usv_frame_desc* frame,
                                        int32_t n_pairs, const int32_t* h_tx, const int32_t* h_ty, int32_t n_templates,
                                        const usv_search_params* params, const usv_outputs* h_out, uint32_t* h_cost_rows,
                                        double* h_score_rows, int32_t row_cap) {
  if (!ctx) return USV_ERR_INVALID_ARG;
  if (!h_tx) return fail(ctx, USV_ERR_INVALID_ARG, "null template list");
  return match_host(ctx, h_left, h_right, frame, n_pairs, params, h_out, h_tx, h_ty, n_templates, h_cost_rows, h_score_rows, row_cap);
}

extern "C" int usv_match_dense_subpixel_host(usv_ctx* ctx, const uint8_t* h_left, const uint8_t* h_right, const usv_frame_desc* frame,
                                             int32_t n_pairs, const usv_search_params* params, const usv_outputs* h_out,
                                             int32_t* h_disparity_x16, double* h_distance) {
  if (!ctx) return USV_ERR_INVALID_ARG;
  usv_outputs none;
  memset(&none, 0, sizeof(none));
  const SubpixelOut sub = {h_disparity_x16, h_distance};
  return match_host(ctx, h_left, h_right, frame, n_pairs, params, h_out ? h_out : &none, nullptr, nullptr, 0, nullptr, nullptr, 0, &sub);
}

// ---- distance family ------------------------------------------------------------------
static int up(usv_ctx* ctx, DevBuf& b, const void* h, size_t bytes) {
  int rc = grow(ctx, b, bytes ? bytes : 16);
  if (rc) return rc;
  if (bytes) CU(cudaMemcpyAsync(b.p, h, bytes, cudaMemcpyHostToDevice, ctx->stream));
  return USV_OK;
}

// ---- ResolveMatchList on the GPU (usv_resolve.cu) ------------------------------------------
static int resolve_device(usv_ctx* ctx, const usv_match* d_in, int64_t n, int32_t skip_unmatched, usv_match* d_out, int64_t cap,
                          int64_t* d_n_out, cudaStream_t st) {
  if (n < 0 || cap < 0 || n >= 0x7fffffffll) return fail(ctx, USV_ERR_INVALID_ARG, "match list length %lld out of range", (long long)n);
  if (!d_n_out || (n > 0 && (!d_in || (cap > 0 && !d_out)))) return fail(ctx, USV_ERR_INVALID_ARG, "null pointer");
  CU(cudaSetDevice(ctx->device));
  const size_t ws = n ? usv::resolve_workspace_bytes(n) : 0;
  int rc = grow(ctx, ctx->resolve_ws, ws ? ws : 16);
  if (rc) return rc;
  int nl = 0;
  cudaError_t e = usv::launch_resolve(d_in, n, skip_unmatched, d_out, cap, (long long*)d_n_out, ctx->resolve_ws.p, ws, st, &nl);
  if (e != cudaSuccess) return fail(ctx, USV_ERR_CUDA, "resolve launch: %s", cudaGetErrorString(e));
  ctx->launches += nl;
  if (nl) ctx->last_kernel = "resolve_next_smaller_kernel";
  return USV_OK;
}

extern "C" int usv_resolve_match_list_device(usv_ctx* ctx, const usv_match* d_in, int64_t n, int32_t skip_unmatched, usv_match* d_out,
                                             int64_t cap, int64_t* d_n_out, void* cuda_stream) {
  if (!ctx) return USV_ERR_INVALID_ARG;
  return resolve_device(ctx, d_in, n, skip_unmatched, d_out, cap, d_n_out, (cudaStream_t)cuda_stream);
}

extern "C" int usv_resolve_match_list(usv_ctx* ctx, const usv_match* h_in, int64_t n, int32_t skip_unmatched, usv_match* h_out,
                                      int64_t cap, int64_t* n_out) {
  if (!ctx) return USV_ERR_INVALID_ARG;
  if (n < 0 || cap < 0 || !n_out || (n > 0 && !h_in) || (cap > 0 && !h_out)) return fail(ctx, USV_ERR_INVALID_ARG, "bad arguments");
  *n_out = 0;
  if (n == 0) return USV_OK;
  CU(cudaSetDevice(ctx->device));
  int rc;
  const int64_t room = cap < n ? cap : n;  // the output is never longer than the input
  if ((rc = up(ctx, ctx->misc[0], h_in, sizeof(usv_match) * (size_t)n))) return rc;
  if ((rc = grow(ctx, ctx->misc[1], sizeof(usv_match) * (size_t)(room ? room : 1)))) return rc;
  if ((rc = grow(ctx, ctx->misc[2], sizeof(int64_t)))) return rc;
  if ((rc = resolve_device(ctx, (const usv_match*)ctx->misc[0].p, n, skip_unmatched, (usv_match*)ctx->misc[1].p, room,
                           (int64_t*)ctx->misc[2].p, ctx->stream)))
    return rc;
  int64_t total = 0;
  CU(cudaMemcpyAsync(&total, ctx->misc[2].p, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  const int64_t m = total < room ? total : room;
  if (m > 0) CU(cudaMemcpy(h_out, ctx->misc[1].p, sizeof(usv_match) * (size_t)m, cudaMemcpyDeviceToHost));
  *n_out = total;
  return USV_OK;
}

// ---- generate -> resolve -> distance in one call, host buffers (the reference's call order, P/Main.cpp:1115-1143) ----
extern "C" int usv_block_search_host(usv_ctx* ctx, const uint8_t* h_left, const uint8_t* h_right, const usv_frame_desc* f,
                                     const usv_search_params* p, usv_match* h_matches, double* h_distance, int64_t cap, int64_t* n_out) {
  if (!ctx) return USV_ERR_INVALID_ARG;
  int rc = check_common(ctx, f, p, 1);
  if (rc) return rc;
  if (!h_left || !h_right || !n_out || cap < 0 || (cap > 0 && !h_matches)) return fail(ctx, USV_ERR_INVALID_ARG, "bad arguments");
  *n_out = 0;
  int32_t nx, ny;
  if (usv_grid_dims(f, p, &nx, &ny, nullptr)) return fail(ctx, USV_ERR_INVALID_ARG, "bad geometry");
  const int64_t n_win = (int64_t)nx * ny;
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  // frames: caller memory -> pinned staging at the device pitch (one host pass; the H2D is then one asynchronous copy
  // per camera) -> HBM
  const usv_frame_desc df = device_frame_desc(f);
  const int row_bytes = f->width * f->channels, pitch = df.row_stride;
  const size_t fbytes = (size_t)df.frame_stride;
  if ((rc = grow(ctx, ctx->pin[0], 2 * fbytes))) return rc;
  uint8_t* stage = (uint8_t*)ctx->pin[0].p;
  for (int k = 0; k < 2; ++k) {
    const uint8_t* src = k ? h_right : h_left;
    uint8_t* dst = stage + k * fbytes;
    if (f->row_stride == pitch) memcpy(dst, src, fbytes);
    else for (int y = 0; y < f->height; ++y) memcpy(dst + (size_t)y * pitch, src + (size_t)y * f->row_stride, row_bytes);
  }
  if ((rc = grow(ctx, ctx->in_l, fbytes)) || (rc = grow(ctx, ctx->in_r, fbytes))) return rc;
  CU(cudaMemcpyAsync(ctx->in_l.p, stage, fbytes, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(ctx->in_r.p, stage + fbytes, fbytes, cudaMemcpyHostToDevice, st));
  // generate (+ per-window first minimum): the winners stay in HBM
  if ((rc = grow(ctx, ctx->out[0], sizeof(usv_match) * n_win))) return rc;
  usv_outputs d_out;
  memset(&d_out, 0, sizeof(d_out));
  d_out.matches = (usv_match*)ctx->out[0].p;
  if ((rc = match_device(ctx, (const uint8_t*)ctx->in_l.p, (const uint8_t*)ctx->in_r.p, &df, 1, p, &d_out, nullptr, nullptr, 0, nullptr,
                         nullptr, 0, st)))
    return rc;
  const char* match_kernel = ctx->last_kernel;
  // resolve: the reference's whole-list greedy pass over the accepted winners (usv_resolve.cu)
  if ((rc = grow(ctx, ctx->misc[1], sizeof(usv_match) * n_win)) || (rc = grow(ctx, ctx->misc[2], sizeof(int64_t)))) return rc;
  if ((rc = resolve_device(ctx, d_out.matches, n_win, 1, (usv_match*)ctx->misc[1].p, n_win, (int64_t*)ctx->misc[2].p, st))) return rc;
  // distance of every surviving match (P/Main.cpp:681-694)
  const bool want_dist = h_distance != nullptr && p->distance_kind != USV_DIST_NONE;
  if (want_dist) {
    const double* lut = nullptr;
    if ((rc = ensure_lut(ctx, p->distance_kind, f->width, st, &lut))) return rc;
    if ((rc = grow(ctx, ctx->misc[3], sizeof(double) * n_win))) return rc;
    CU(usv::launch_match_list_distance((const usv_match*)ctx->misc[1].p, (const long long*)ctx->misc[2].p, n_win, nx, p->stride_x,
                                       f->width - p->tmpl_w + 1, p->camera_side, p->distance_kind, lut, ctx->lut_n[p->distance_kind],
                                       (double*)ctx->misc[3].p, st));
    ctx->launches++;
  }
  ctx->last_kernel = match_kernel;
  // results: count first, then exactly the surviving records through pinned staging
  if ((rc = grow(ctx, ctx->pin[1], sizeof(usv_match) * n_win + 64)) || (rc = grow(ctx, ctx->pin[2], sizeof(double) * n_win + 64))) return rc;
  int64_t* h_n = (int64_t*)((uint8_t*)ctx->pin[1].p + sizeof(usv_match) * n_win);
  CU(cudaMemcpyAsync(h_n, ctx->misc[2].p, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  const int64_t total = *h_n, m = total < cap ? total : cap;
  if (m > 0) {
    CU(cudaMemcpyAsync(ctx->pin[1].p, ctx->misc[1].p, sizeof(usv_match) * (size_t)m, cudaMemcpyDeviceToHost, st));
    if (want_dist) CU(cudaMemcpyAsync(ctx->pin[2].p, ctx->misc[3].p, sizeof(double) * (size_t)m, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    memcpy(h_matches, ctx->pin[1].p, sizeof(usv_match) * (size_t)m);
    if (want_dist) memcpy(h_distance, ctx->pin[2].p, sizeof(double) * (size_t)m);
    else if (h_distance) memset(h_distance, 0, sizeof(double) * (size_t)m);
  }
  *n_out = total;
  return check_dev_status(ctx);
}

// ---- pre-pass (usv_preprocess.cu) -------------------------------------------------------------
static int preprocess_check(usv_ctx* ctx, int32_t n_frames, const usv_preprocess_params* p, const void* map1, const void* map2) {
  if (!p) return fail(ctx, USV_ERR_INVALID_ARG, "null params");
  if (n_frames < 0) return fail(ctx, USV_ERR_INVALID_ARG, "n_frames < 0");
  if (p->width <= 0 || p->height <= 0 || p->width > 32767 || p->height > 32767) return fail(ctx, USV_ERR_INVALID_ARG, "bad frame size");
  if (p->src_stride < 3 * p->width || p->dst_stride < p->width) return fail(ctx, USV_ERR_INVALID_ARG, "stride smaller than a row");
  if (n_frames > 1 && (p->src_frame_stride < (int64_t)p->src_stride * p->height || p->dst_frame_stride < (int64_t)p->dst_stride * p->height))
    return fail(ctx, USV_ERR_INVALID_ARG, "frame stride smaller than a frame");
  if (p->flavour != USV_PRE_OPENCV3 && p->flavour != USV_PRE_OPENCV4) return fail(ctx, USV_ERR_INVALID_ARG, "unknown flavour %d", p->flavour);
  if ((map1 == nullptr) != (map2 == nullptr)) return fail(ctx, USV_ERR_INVALID_ARG, "map1 and map2 come as a pair");
  return USV_OK;
}

extern "C" int usv_preprocess_device(usv_ctx* ctx, const uint8_t* d_bgr, int32_t n_frames, const int16_t* d_map1, const uint16_t* d_map2,
                                     const usv_preprocess_params* p, uint8_t* d_gray, void* cuda_stream) {
  if (!ctx) return USV_ERR_INVALID_ARG;
  int rc = preprocess_check(ctx, n_frames, p, d_map1, d_map2);
  if (rc) return rc;
  if (n_frames == 0) return USV_OK;
  if (!d_bgr || !d_gray) return fail(ctx, USV_ERR_INVALID_ARG, "null device pointer");
  CU(cudaSetDevice(ctx->device));
  if (p->lighting && (rc = grow(ctx, ctx->pre_ws, usv::preprocess_scratch_bytes(p->width, p->height, n_frames)))) return rc;
  int nl = 0;
  cudaError_t e = usv::launch_preprocess(ctx->device, d_bgr, d_gray, d_map1, d_map2, n_frames, p->width, p->height, p->src_stride,
                                         p->dst_stride, p->src_frame_stride, p->dst_frame_stride, p->flavour, p->lighting,
                                         ctx->pre_ws.p, (cudaStream_t)cuda_stream, &nl);
  if (e != cudaSuccess) return fail(ctx, USV_ERR_CUDA, "preprocess launch: %s", cudaGetErrorString(e));
  ctx->launches += nl;
  ctx->last_kernel = p->lighting ? "rectify_hsv_hist_kernel+equalize_lut_kernel+hsv_gray_kernel" : "rectify_gray_kernel";
  return USV_OK;
}

// `n` frames of `height` rows of `row_bytes` between host and device buffers of the same layout (rows `stride` apart,
// frames `frame_stride` apart): only those bytes are read and written, never a row's padding or the gap between two
// frames, which belong to the caller. One 2D copy when the frames are packed, one per frame otherwise.
static int copy_frame_bytes(usv_ctx* ctx, uint8_t* dst, const uint8_t* src, int32_t n, int row_bytes, int height, int stride,
                            int64_t frame_stride, cudaMemcpyKind kind) {
  if (n == 1 || frame_stride == (int64_t)stride * height) {
    CU(cudaMemcpy2DAsync(dst, stride, src, stride, row_bytes, (size_t)height * n, kind, ctx->stream));
  } else {
    for (int32_t i = 0; i < n; ++i)
      CU(cudaMemcpy2DAsync(dst + (size_t)i * frame_stride, stride, src + (size_t)i * frame_stride, stride, row_bytes, height, kind,
                           ctx->stream));
  }
  return USV_OK;
}

extern "C" int usv_preprocess_host(usv_ctx* ctx, const uint8_t* h_bgr, int32_t n_frames, const int16_t* h_map1, const uint16_t* h_map2,
                                   const usv_preprocess_params* p, uint8_t* h_gray) {
  if (!ctx) return USV_ERR_INVALID_ARG;
  int rc = preprocess_check(ctx, n_frames, p, h_map1, h_map2);
  if (rc) return rc;
  if (n_frames == 0) return USV_OK;
  if (!h_bgr || !h_gray) return fail(ctx, USV_ERR_INVALID_ARG, "null host pointer");
  CU(cudaSetDevice(ctx->device));
  // the device copies keep the caller's layout; only the frames' own bytes cross the bus
  const size_t src_bytes = (size_t)(n_frames - 1) * p->src_frame_stride + (size_t)p->src_stride * p->height;
  const size_t dst_bytes = (size_t)(n_frames - 1) * p->dst_frame_stride + (size_t)p->dst_stride * p->height;
  const size_t px = (size_t)p->width * p->height;
  if ((rc = grow(ctx, ctx->misc[0], src_bytes)) ||
      (rc = copy_frame_bytes(ctx, (uint8_t*)ctx->misc[0].p, h_bgr, n_frames, 3 * p->width, p->height, p->src_stride,
                             p->src_frame_stride, cudaMemcpyHostToDevice)))
    return rc;
  if ((rc = grow(ctx, ctx->misc[1], dst_bytes))) return rc;
  if (h_map1) {
    if ((rc = up(ctx, ctx->misc[2], h_map1, px * 4))) return rc;
    if ((rc = up(ctx, ctx->misc[3], h_map2, px * 2))) return rc;
  }
  rc = usv_preprocess_device(ctx, (const uint8_t*)ctx->misc[0].p, n_frames, h_map1 ? (const int16_t*)ctx->misc[2].p : nullptr,
                             h_map1 ? (const uint16_t*)ctx->misc[3].p : nullptr, p, (uint8_t*)ctx->misc[1].p, ctx->stream);
  if (rc) return rc;
  if ((rc = copy_frame_bytes(ctx, h_gray, (const uint8_t*)ctx->misc[1].p, n_frames, p->width, p->height, p->dst_stride,
                             p->dst_frame_stride, cudaMemcpyDeviceToHost)))
    return rc;
  CU(cudaStreamSynchronize(ctx->stream));
  return USV_OK;
}

extern "C" int usv_id_matcher(usv_ctx* ctx, const usv_match* h_cur, int64_t n_cur, const usv_match* h_old, int64_t n_old,
                              int32_t* h_out3, int64_t cap, int64_t* n_out) {
  if (!ctx) return USV_ERR_INVALID_ARG;
  if (n_cur < 0 || n_old < 0 || cap < 0 || !n_out || (n_cur > 0 && !h_cur) || (n_old > 0 && !h_old) || (cap > 0 && !h_out3) ||
      n_cur >= 0x7fffffffll || n_old >= 0x7fffffffll)
    return fail(ctx, USV_ERR_INVALID_ARG, "bad arguments");
  *n_out = 0;
  if (n_cur == 0 || n_old == 0) return USV_OK;  // P/Main.cpp:487-489
  CU(cudaSetDevice(ctx->device));
  int rc;
  if ((rc = up(ctx, ctx->misc[0], h_cur, sizeof(usv_match) * (size_t)n_cur))) return rc;
  if ((rc = up(ctx, ctx->misc[1], h_old, sizeof(usv_match) * (size_t)n_old))) return rc;
  if ((rc = grow(ctx, ctx->misc[2], sizeof(int32_t) * 3 * (size_t)(cap ? cap : 1)))) return rc;
  if ((rc = grow(ctx, ctx->misc[3], sizeof(int64_t)))) return rc;
  const size_t ws = usv::id_matcher_workspace_bytes(n_cur);
  if ((rc = grow(ctx, ctx->resolve_ws, ws))) return rc;
  cudaError_t e = usv::launch_id_matcher((const usv_match*)ctx->misc[0].p, n_cur, (const usv_match*)ctx->misc[1].p, n_old,
                                         (int*)ctx->misc[2].p, cap, (long long*)ctx->misc[3].p, ctx->resolve_ws.p, ws, ctx->stream);
  if (e != cudaSuccess) return fail(ctx, USV_ERR_CUDA, "id_matcher launch: %s", cudaGetErrorString(e));
  ctx->launches += 2;
  ctx->last_kernel = "id_matcher_write_kernel";
  int64_t total = 0;
  CU(cudaMemcpyAsync(&total, ctx->misc[3].p, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  const int64_t m = total < cap ? total : cap;
  if (m > 0) CU(cudaMemcpy(h_out3, ctx->misc[2].p, sizeof(int32_t) * 3 * (size_t)m, cudaMemcpyDeviceToHost));
  *n_out = total;
  return USV_OK;
}

extern "C" int usv_distance_lut(usv_ctx* ctx, int32_t kind, int32_t n, double* h_lut) {
  if (!ctx) return USV_ERR_INVALID_ARG;
  if (n <= 0 || !h_lut) return fail(ctx, USV_ERR_INVALID_ARG, "bad arguments");
  if (kind != USV_DIST_PINHOLE && kind != USV_DIST_POWERLAW) return fail(ctx, USV_ERR_INVALID_ARG, "unknown distance_kind %d", kind);
  CU(cudaSetDevice(ctx->device));
  const double* lut = nullptr;
  int rc = ensure_lut(ctx, kind, n, ctx->stream, &lut);  // the table the kernels' epilogue reads
  if (rc) return rc;
  CU(cudaMemcpyAsync(h_lut, lut, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return USV_OK;
}

extern "C" int usv_disparity_to_distance(usv_ctx* ctx, const int32_t* h_disp, int64_t n, int32_t kind, double* h_dist) {
  if (!ctx) return USV_ERR_INVALID_ARG;
  if (n < 0 || (n > 0 && (!h_disp || !h_dist))) return fail(ctx, USV_ERR_INVALID_ARG, "bad arguments");
  if (kind != USV_DIST_PINHOLE && kind != USV_DIST_POWERLAW) return fail(ctx, USV_ERR_INVALID_ARG, "unknown distance_kind %d", kind);
  if (n == 0) return USV_OK;
  CU(cudaSetDevice(ctx->device));
  int rc;
  if ((rc = up(ctx, ctx->misc[0], h_disp, sizeof(int32_t) * n))) return rc;
  if ((rc = grow(ctx, ctx->misc[1], sizeof(double) * n))) return rc;
  CU(usv::launch_disparity_to_distance((const int*)ctx->misc[0].p, n, kind, (double*)ctx->misc[1].p, ctx->stream));
  ctx->launches++;
  CU(cudaMemcpyAsync(h_dist, ctx->misc[1].p, sizeof(double) * n, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return USV_OK;
}

extern "C" int usv_moving_object_distance(usv_ctx* ctx, int32_t camera_side, int64_t t_this_ns, const float* this_xy, int32_t n_this,
                                          const float* other_xy, int32_t n_other, const float* old_xy, int32_t n_old,
                                          const float* older_xy, int32_t n_older, const int32_t* idx3, int32_t n_idx,
                                          int64_t t_other_ns, int64_t t_old_ns, int64_t t_older_ns, double* h_dist, int32_t* n_out) {
  if (!ctx) return USV_ERR_INVALID_ARG;
  if (n_this < 0 || n_other < 0 || n_old < 0 || n_older < 0 || n_idx < 0) return fail(ctx, USV_ERR_INVALID_ARG, "negative count");
  if (n_out) *n_out = 0;
  // P/DistanceCalculator.cpp:28 — nothing is produced unless all three histories are non-empty
  if (n_other == 0 || n_old == 0 || n_older == 0 || n_idx == 0) return USV_OK;
  if (!other_xy || !old_xy || !older_xy || !idx3 || !h_dist || (n_this > 0 && !this_xy))
    return fail(ctx, USV_ERR_INVALID_ARG, "null pointer");
  CU(cudaSetDevice(ctx->device));
  int rc;
  if ((rc = up(ctx, ctx->misc[0], this_xy, sizeof(float) * 2 * n_this))) return rc;
  if ((rc = up(ctx, ctx->misc[1], other_xy, sizeof(float) * 2 * n_other))) return rc;
  if ((rc = up(ctx, ctx->misc[2], old_xy, sizeof(float) * 2 * n_old))) return rc;
  if ((rc = up(ctx, ctx->misc[3], older_xy, sizeof(float) * 2 * n_older))) return rc;
  if ((rc = up(ctx, ctx->misc[4], idx3, sizeof(int32_t) * 3 * n_idx))) return rc;
  if ((rc = grow(ctx, ctx->misc[5], sizeof(double) * n_idx))) return rc;
  CU(usv::launch_moving_object_distance(camera_side, t_this_ns, (const float*)ctx->misc[0].p, n_this, (const float*)ctx->misc[1].p,
                                        n_other, (const float*)ctx->misc[2].p, n_old, (const float*)ctx->misc[3].p, n_older,
                                        (const int*)ctx->misc[4].p, n_idx, t_other_ns, t_old_ns, t_older_ns,
                                        (double*)ctx->misc[5].p, ctx->stream));
  ctx->launches++;
  CU(cudaMemcpyAsync(h_dist, ctx->misc[5].p, sizeof(double) * n_idx, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  if (n_out) *n_out = n_idx;
  return USV_OK;
}

extern "C" int usv_coordinate_position(usv_ctx* ctx, int32_t camera_side, const double* h_dist, const float* h_xy, int64_t n,
                                       double* h_xyz) {
  if (!ctx) return USV_ERR_INVALID_ARG;
  if (n < 0 || (n > 0 && (!h_dist || !h_xy || !h_xyz))) return fail(ctx, USV_ERR_INVALID_ARG, "bad arguments");
  if (n == 0) return USV_OK;
  CU(cudaSetDevice(ctx->device));
  int rc;
  if ((rc = up(ctx, ctx->misc[0], h_dist, sizeof(double) * n))) return rc;
  if ((rc = up(ctx, ctx->misc[1], h_xy, sizeof(float) * 2 * n))) return rc;
  if ((rc = grow(ctx, ctx->misc[2], sizeof(double) * 3 * n))) return rc;
  CU(usv::launch_coordinate_position(camera_side, (const double*)ctx->misc[0].p, (const float*)ctx->misc[1].p, n,
                                     (double*)ctx->misc[2].p, ctx->stream));
  ctx->launches++;
  CU(cudaMemcpyAsync(h_xyz, ctx->misc[2].p, sizeof(double) * 3 * n, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return USV_OK;
}

// ---- the reference's original contour cost (matchShapes I1 + area ratio), P/Main.cpp:403-426 ----
extern "C" int usv_match_contours(usv_ctx* ctx, const int32_t* pts_this, const int32_t* off_this, int32_t n_this,
                                  const int32_t* pts_other, const int32_t* off_other, int32_t n_other, double accept_threshold,
                                  usv_match* h_out, int64_t cap, int64_t* n_out, double* h_cost_matrix) {
  if (!ctx) return USV_ERR_INVALID_ARG;
  if (n_out) *n_out = 0;
  if (n_this < 0 || n_other < 0 || cap < 0) return fail(ctx, USV_ERR_INVALID_ARG, "negative count");
  if (n_this == 0 || n_other == 0) return USV_OK;  // P/Main.cpp:405
  if (!pts_this || !off_this || !pts_other || !off_other || (cap > 0 && !h_out)) return fail(ctx, USV_ERR_INVALID_ARG, "null pointer");
  for (int i = 0; i < n_this; ++i) if (off_this[i + 1] < off_this[i]) return fail(ctx, USV_ERR_INVALID_ARG, "offsets must ascend");
  for (int i = 0; i < n_other; ++i) if (off_other[i + 1] < off_other[i]) return fail(ctx, USV_ERR_INVALID_ARG, "offsets must ascend");
  CU(cudaSetDevice(ctx->device));
  int rc;
  const size_t np_l = (size_t)off_this[n_this], np_r = (size_t)off_other[n_other];
  if ((rc = up(ctx, ctx->misc[0], pts_this, sizeof(int32_t) * 2 * np_l))) return rc;
  if ((rc = up(ctx, ctx->misc[1], off_this, sizeof(int32_t) * (n_this + 1)))) return rc;
  if ((rc = up(ctx, ctx->misc[2], pts_other, sizeof(int32_t) * 2 * np_r))) return rc;
  if ((rc = up(ctx, ctx->misc[3], off_other, sizeof(int32_t) * (n_other + 1)))) return rc;
  if ((rc = grow(ctx, ctx->misc[4], sizeof(double) * 8 * n_this))) return rc;
  if ((rc = grow(ctx, ctx->misc[5], sizeof(double) * 8 * n_other))) return rc;
  const size_t n_pairs = (size_t)n_this * n_other;
  if ((rc = grow(ctx, ctx->misc[6], sizeof(double) * n_pairs))) return rc;
  CU(usv::launch_contour_descriptors((const int*)ctx->misc[0].p, (const int*)ctx->misc[1].p, n_this, (double*)ctx->misc[4].p, ctx->stream));
  CU(usv::launch_contour_descriptors((const int*)ctx->misc[2].p, (const int*)ctx->misc[3].p, n_other, (double*)ctx->misc[5].p, ctx->stream));
  CU(usv::launch_contour_costs((const double*)ctx->misc[4].p, n_this, (const double*)ctx->misc[5].p, n_other, (double*)ctx->misc[6].p, ctx->stream));
  ctx->launches += 3;
  ctx->last_kernel = "contour_cost_kernel";
  std::vector<double> cost(n_pairs);
  CU(cudaMemcpyAsync(cost.data(), ctx->misc[6].p, sizeof(double) * n_pairs, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  if (h_cost_matrix) memcpy(h_cost_matrix, cost.data(), sizeof(double) * n_pairs);
  int64_t n = 0;
  for (int i = 0; i < n_this; ++i)      // i-major (P/Main.cpp:408)
    for (int j = 0; j < n_other; ++j) { // j-minor (P/Main.cpp:410)
      const double v = cost[(size_t)i * n_other + j];
      if (v < accept_threshold) {       // Is it at least a partial match? (P/Main.cpp:417); NaN never passes
        if (n >= cap) return fail(ctx, USV_ERR_INVALID_ARG, "output capacity %lld too small", (long long)cap);
        h_out[n].LeftIndex = (uint32_t)i; h_out[n].RightIndex = (uint32_t)j; h_out[n].MatchValue = v;
        ++n;
      }
    }
  if (n_out) *n_out = n;
  return USV_OK;
}

// ---- roofline denominator: sustained issue rate of the packed-byte integer instruction ----
extern "C" int usv_probe_issue_rate(usv_ctx* ctx, int32_t which, double target_ms, double* lane_inst_per_s) {
  if (!ctx) return USV_ERR_INVALID_ARG;
  if (!lane_inst_per_s || which < 0 || which > 1 || !(target_ms > 0)) return fail(ctx, USV_ERR_INVALID_ARG, "bad arguments");
  CU(cudaSetDevice(ctx->device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, ctx->device));
  int rc = grow(ctx, ctx->misc[7], 64);
  if (rc) return rc;
  CU(usv::run_issue_probe(which, prop.multiProcessorCount, target_ms, lane_inst_per_s, (uint32_t*)ctx->misc[7].p, ctx->stream));
  ctx->launches += 3;
  return USV_OK;
}

// ---- nearest-timestamp pairing (pure host, O(nL + nR)) ---------------------------------
extern "C" int64_t usv_pair_nearest(const double* tl, int64_t nl, const double* tr, int64_t nr, double max_dt, int32_t* out_l,
                                    int32_t* out_r, int64_t cap) {
  if (nl < 0 || nr < 0 || cap < 0 || (nl > 0 && !tl) || (nr > 0 && !tr) || (cap > 0 && (!out_l || !out_r))) return USV_ERR_INVALID_ARG;
  if (nl > INT32_MAX || nr > INT32_MAX) return USV_ERR_INVALID_ARG;
  for (int64_t i = 1; i < nl; ++i) if (tl[i] < tl[i - 1]) return USV_ERR_INVALID_ARG;  // must be ascending
  for (int64_t i = 1; i < nr; ++i) if (tr[i] < tr[i - 1]) return USV_ERR_INVALID_ARG;
  int64_t n = 0, p = 0;
  // group state: left frames that picked the same right frame are contiguous
  int64_t g_right = -1, g_left = -1;
  double g_gap = 0.0;
  auto flush = [&]() -> bool {
    if (g_right < 0) return true;
    if (n >= cap) return false;
    out_l[n] = (int32_t)g_left; out_r[n] = (int32_t)g_right; ++n;
    g_right = -1;
    return true;
  };
  for (int64_t i = 0; i < nl && nr > 0; ++i) {
    while (p < nr && tr[p] < tl[i]) ++p;  // p = first right frame at or after tl[i]
    int64_t pick; double gap;
    if (p == 0) { pick = 0; gap = std::fabs(tl[i] - tr[0]); }
    else {
      int64_t q = p - 1;
      while (q > 0 && tr[q - 1] == tr[q]) --q;  // lowest index among equal timestamps
      double a = std::fabs(tl[i] - tr[q]);
      if (p < nr) {
        double b = std::fabs(tl[i] - tr[p]);
        if (b < a) { pick = p; gap = b; } else { pick = q; gap = a; }  // earlier frame on a tie
      } else { pick = q; gap = a; }
    }
    if (!(gap <= max_dt)) continue;
    if (pick == g_right) {
      if (gap < g_gap) { g_left = i; g_gap = gap; }  // the closer left frame keeps it (lowest index on a tie)
    } else {
      if (!flush()) return USV_ERR_INVALID_ARG;
      g_right = pick; g_left = i; g_gap = gap;
    }
  }
  if (!flush()) return USV_ERR_INVALID_ARG;
  return n;
}

// ---- streamed matching -------------------------------------------------------------------
struct Slot {
  cudaStream_t st = nullptr;
  cudaEvent_t done = nullptr;
  PinnedBuf h_l, h_r;
  DevBuf d_l, d_r;
  PinnedBuf h_arr[kNumOut];  // the arrays of the output mask; h_out and d_out point at them
  DevBuf d_arr[kNumOut];
  usv_outputs h_out{}, d_out{};
  DevBuf corr_ws;  // planes + window statistics of the sliding correlation kernel: per slot, the slots run concurrently
  DevBuf win_ws;   // winners (RightIndex + value) for the resolved disparity map when the caller did not ask for them
  Slot() = default;
  Slot(const Slot&) = delete;
  Slot& operator=(const Slot&) = delete;
  ~Slot() {
    if (done) cudaEventDestroy(done);
    if (st) cudaStreamDestroy(st);
  }
};

struct usv_stream {
  usv_ctx* ctx = nullptr;
  int device = 0;
  usv_frame_desc fd;  // layout of the slots' pinned frames and of their device frames (the same: one copy per camera)
  usv_search_params params;
  int32_t pairs_per_slot = 0, n_slots = 0;
  uint32_t mask = 0;
  int64_t n_win = 0;
  std::unique_ptr<Slot[]> slots;
};

extern "C" int usv_stream_destroy(usv_stream* s) {
  if (!s) return USV_ERR_INVALID_ARG;
  cudaSetDevice(s->device);
  for (int i = 0; i < s->n_slots; ++i)
    if (s->slots[i].st) cudaStreamSynchronize(s->slots[i].st);
  usv_ctx* ctx = s->ctx;
  delete s;
  if (ctx) ctx->open_streams--;
  return USV_OK;
}

extern "C" int usv_stream_create(usv_ctx* ctx, const usv_frame_desc* frame, const usv_search_params* params, int32_t pairs_per_slot,
                                 int32_t n_slots, uint32_t output_mask, usv_stream** out) {
  if (!ctx || !out) return USV_ERR_INVALID_ARG;
  *out = nullptr;
  if (pairs_per_slot <= 0 || n_slots <= 0 || n_slots > 64) return fail(ctx, USV_ERR_INVALID_ARG, "bad slot geometry");
  int rc = check_common(ctx, frame, params, pairs_per_slot);
  if (rc) return rc;
  if ((output_mask & USV_OUT_RAW_COST_U16) && (rc = check_cost_u16(ctx, frame, params))) return rc;
  int32_t nx, ny;
  if (usv_grid_dims(frame, params, &nx, &ny, nullptr)) return fail(ctx, USV_ERR_INVALID_ARG, "bad geometry");
  CU(cudaSetDevice(ctx->device));
  usv_stream* s = new (std::nothrow) usv_stream();
  if (!s) return fail(ctx, USV_ERR_NOMEM, "out of host memory");
  s->ctx = ctx; s->device = ctx->device; ctx->open_streams++; s->params = *params; s->pairs_per_slot = pairs_per_slot; s->n_slots = n_slots; s->mask = output_mask;
  s->n_win = (int64_t)nx * ny;
  // pinned staging keeps the frames tightly packed at the device layout, so each slot needs exactly one
  // cudaMemcpyAsync per camera
  s->fd = device_frame_desc(frame);
  s->slots.reset(new Slot[n_slots]);
  const size_t fbytes = (size_t)s->fd.frame_stride * pairs_per_slot;
  const size_t n_res = (size_t)s->n_win * pairs_per_slot;
  cudaError_t e = cudaSuccess;
  for (int k = 0; k < n_slots && e == cudaSuccess; ++k) {
    Slot& sl = s->slots[k];
    if ((e = cudaStreamCreateWithFlags(&sl.st, cudaStreamNonBlocking)) != cudaSuccess) break;
    if ((e = cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming)) != cudaSuccess) break;
    if ((e = sl.h_l.alloc(fbytes)) != cudaSuccess || (e = sl.h_r.alloc(fbytes)) != cudaSuccess) break;
    if ((e = sl.d_l.alloc(fbytes)) != cudaSuccess || (e = sl.d_r.alloc(fbytes)) != cudaSuccess) break;
    memset(sl.h_l.p, 0, fbytes);
    memset(sl.h_r.p, 0, fbytes);
    for (int i = 0; i < kNumOut; ++i) {
      if (!(output_mask & (1u << i))) continue;
      if ((e = sl.h_arr[i].alloc(kOutElem[i] * n_res)) != cudaSuccess || (e = sl.d_arr[i].alloc(kOutElem[i] * n_res)) != cudaSuccess) break;
      *out_slot(&sl.h_out, i) = sl.h_arr[i].p;
      *out_slot(&sl.d_out, i) = sl.d_arr[i].p;
    }
  }
  if (e != cudaSuccess) {
    fail(ctx, USV_ERR_NOMEM, "stream allocation: %s", cudaGetErrorString(e));
    usv_stream_destroy(s);
    return USV_ERR_NOMEM;
  }
  *out = s;
  return USV_OK;
}

extern "C" int usv_stream_slot(usv_stream* s, int32_t slot, uint8_t** h_left, uint8_t** h_right, usv_outputs* h_out) {
  if (!s || slot < 0 || slot >= s->n_slots) return USV_ERR_INVALID_ARG;
  if (h_left) *h_left = (uint8_t*)s->slots[slot].h_l.p;
  if (h_right) *h_right = (uint8_t*)s->slots[slot].h_r.p;
  if (h_out) *h_out = s->slots[slot].h_out;
  return USV_OK;
}

extern "C" int usv_stream_frame_desc(const usv_stream* s, usv_frame_desc* out) {
  if (!s || !out) return USV_ERR_INVALID_ARG;
  *out = s->fd;
  return USV_OK;
}

static int check_host_frame(usv_stream* s, const usv_frame_desc* hf) {
  if (hf->width != s->fd.width || hf->height != s->fd.height || hf->channels != s->fd.channels ||
      hf->row_stride < hf->width * hf->channels)
    return fail(s->ctx, USV_ERR_INVALID_ARG, "frame geometry differs from the stream's");
  if (hf->frame_stride < (int64_t)hf->row_stride * hf->height)
    return fail(s->ctx, USV_ERR_INVALID_ARG, "frame_stride %lld smaller than one frame", (long long)hf->frame_stride);
  return USV_OK;
}

// the frames of one submit: pair i is frame idx_left[i] of `left` and frame idx_right[i] of `right` (frame i of each
// without index arrays), laid out per `hf`
struct FrameSrc {
  const uint8_t* left;
  const uint8_t* right;
  const usv_frame_desc* hf;
  const int32_t* idx_left = nullptr;
  const int32_t* idx_right = nullptr;
  int64_t n_store = 0;  // frames of each store, with index arrays
};

// frames H2D, kernels, results D2H (into the caller's h_dst instead of the slot's pinned arrays when given) and the
// completion event of one slot, all on its stream
static int submit(usv_stream* s, int32_t slot, int32_t n_pairs, const FrameSrc& src, const usv_outputs* h_dst) {
  usv_ctx* ctx = s->ctx;
  if (n_pairs < 0 || n_pairs > s->pairs_per_slot) return fail(ctx, USV_ERR_INVALID_ARG, "n_pairs %d exceeds the slot", n_pairs);
  int rc = check_host_frame(s, src.hf);
  if (rc) return rc;
  const int32_t* idx[2] = {src.idx_left, src.idx_right};
  if (idx[0])
    for (int i = 0; i < n_pairs; ++i)
      if (idx[0][i] < 0 || idx[0][i] >= src.n_store || idx[1][i] < 0 || idx[1][i] >= src.n_store)
        return fail(ctx, USV_ERR_INVALID_ARG, "pair %d: frame index outside the store", i);
  Slot& sl = s->slots[slot];
  usv_outputs dst = h_dst ? *h_dst : sl.h_out;
  if (h_dst)
    for (int i = 0; i < kNumOut; ++i)
      if (((s->mask >> i) & 1u) && !*out_slot(&dst, i)) return fail(ctx, USV_ERR_INVALID_ARG, "destination of output %d of the stream's mask is null", i);
  CU(cudaSetDevice(ctx->device));
  const uint8_t* store[2] = {src.left, src.right};
  uint8_t* d_frames[2] = {(uint8_t*)sl.d_l.p, (uint8_t*)sl.d_r.p};
  for (int k = 0; k < 2; ++k) {
    // runs of consecutive store frames travel as one copy (paired unsynchronised streams are mostly consecutive)
    for (int i = 0; i < n_pairs;) {
      int j = i + 1;
      while (j < n_pairs && (!idx[k] || idx[k][j] == idx[k][j - 1] + 1)) ++j;
      const uint8_t* first = store[k] + (size_t)(idx[k] ? idx[k][i] : i) * src.hf->frame_stride;
      if ((rc = copy_frames(ctx, d_frames[k] + (size_t)i * s->fd.frame_stride, s->fd, first, src.hf, j - i, sl.st))) return rc;
      i = j;
    }
  }
  if (n_pairs > 0) {
    rc = match_device(ctx, d_frames[0], d_frames[1], &s->fd, n_pairs, &s->params, &sl.d_out, nullptr, nullptr, 0, nullptr, nullptr, 0,
                      sl.st, &sl.corr_ws, &sl.win_ws);
    if (rc) return rc;
    const size_t n_res = (size_t)s->n_win * n_pairs;
    for (int i = 0; i < kNumOut; ++i)
      if (*out_slot(&sl.h_out, i))
        CU(cudaMemcpyAsync(*out_slot(&dst, i), *out_slot(&sl.d_out, i), kOutElem[i] * n_res, cudaMemcpyDeviceToHost, sl.st));
  }
  CU(cudaEventRecord(sl.done, sl.st));
  return USV_OK;
}

extern "C" int usv_stream_submit(usv_stream* s, int32_t slot, int32_t n_pairs) {
  if (!s || slot < 0 || slot >= s->n_slots) return USV_ERR_INVALID_ARG;
  const Slot& sl = s->slots[slot];
  return submit(s, slot, n_pairs, {(const uint8_t*)sl.h_l.p, (const uint8_t*)sl.h_r.p, &s->fd}, nullptr);
}

extern "C" int usv_stream_submit_from(usv_stream* s, int32_t slot, const uint8_t* h_left, const uint8_t* h_right,
                                      const usv_frame_desc* hf, int32_t n_pairs) {
  if (!s || slot < 0 || slot >= s->n_slots) return USV_ERR_INVALID_ARG;
  if (!h_left || !h_right || !hf) return fail(s->ctx, USV_ERR_INVALID_ARG, "null pointer");
  return submit(s, slot, n_pairs, {h_left, h_right, hf}, nullptr);
}

extern "C" int usv_stream_submit_gather(usv_stream* s, int32_t slot, const uint8_t* left_store, const int32_t* idx_left,
                                        const uint8_t* right_store, const int32_t* idx_right, int64_t n_store_frames,
                                        const usv_frame_desc* hf, int32_t n_pairs) {
  if (!s || slot < 0 || slot >= s->n_slots) return USV_ERR_INVALID_ARG;
  if (!left_store || !right_store || !idx_left || !idx_right || !hf) return fail(s->ctx, USV_ERR_INVALID_ARG, "null pointer");
  return submit(s, slot, n_pairs, {left_store, right_store, hf, idx_left, idx_right, n_store_frames}, nullptr);
}

extern "C" int usv_stream_submit_io(usv_stream* s, int32_t slot, const uint8_t* h_left, const uint8_t* h_right, const usv_frame_desc* hf,
                                    int32_t n_pairs, const usv_outputs* h_dst) {
  if (!s || slot < 0 || slot >= s->n_slots) return USV_ERR_INVALID_ARG;
  if (!h_left || !h_right || !hf || !h_dst) return fail(s->ctx, USV_ERR_INVALID_ARG, "null pointer");
  return submit(s, slot, n_pairs, {h_left, h_right, hf}, h_dst);
}

extern "C" int usv_host_register(usv_ctx* ctx, void* p, size_t bytes) {
  if (!ctx) return USV_ERR_INVALID_ARG;
  if (!p || bytes == 0) return fail(ctx, USV_ERR_INVALID_ARG, "null buffer");
  CU(cudaSetDevice(ctx->device));
  CU(cudaHostRegister(p, bytes, cudaHostRegisterPortable));
  return USV_OK;
}

extern "C" int usv_host_unregister(usv_ctx* ctx, void* p) {
  if (!ctx) return USV_ERR_INVALID_ARG;
  if (!p) return fail(ctx, USV_ERR_INVALID_ARG, "null buffer");
  CU(cudaHostUnregister(p));
  return USV_OK;
}

extern "C" int usv_stream_wait(usv_stream* s, int32_t slot) {
  if (!s || slot < 0 || slot >= s->n_slots) return USV_ERR_INVALID_ARG;
  usv_ctx* ctx = s->ctx;
  CU(cudaEventSynchronize(s->slots[slot].done));
  return check_dev_status(ctx);
}

extern "C" int usv_stream_bytes_per_pair(const usv_stream* s, int64_t* h2d, int64_t* d2h) {
  if (!s) return USV_ERR_INVALID_ARG;
  if (h2d) *h2d = 2 * s->fd.frame_stride;
  int64_t o = 0;
  for (int i = 0; i < kNumOut; ++i)
    if (s->mask & (1u << i)) o += (int64_t)kOutElem[i] * s->n_win;
  if (d2h) *d2h = o;
  return USV_OK;
}
