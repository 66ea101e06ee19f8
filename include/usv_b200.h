/*
 * usv_b200.h — C-ABI of the B200-native stereo block-search path.
 *
 * This is the drop-in seam underneath the reference's C++ interfaces
 * (`Match`, `GenerateMatchingList`/`ResolveMatchList`, `DistanceCalculator`).
 * Everything is `extern "C"`, plain pointers and sizes; no C++/torch types.
 * Every entry point returns an `int` status (0 = ok, <0 = error) and never
 * throws — the reference's thread entry points use the same 0 / -1 convention
 * (reference P/Main.cpp:818-820, 908-911).
 *
 * Reference items each group replaces (P/ = Unsynchronized_Stereo_Vision_Proj325/):
 *   usv_match                      -> class Match                       P/Match.hpp:4-12
 *   usv_match_dense_* / _templates -> GenerateMatchingList (all-pairs   P/Main.cpp:403-426
 *                                     scoring, i-major / j-minor)  and
 *                                     ResolveMatchList (strict-'>' =    P/Main.cpp:432-477
 *                                     earliest minimum wins, :451)
 *   usv_search_params.accept_*     -> `DMatchValue < 0.75` accept test  P/Main.cpp:417
 *   distance_kind PINHOLE          -> inline disparity + pinhole        P/Main.cpp:681-694
 *   distance_kind POWERLAW         -> power-law fit                     P/DistanceCalculator.cpp:84
 *   usv_resolve_match_list         -> ResolveMatchList (whole list)     P/Main.cpp:432-477
 *   usv_id_matcher                 -> IDMatcher                         P/Main.cpp:483-499
 *   usv_preprocess_*               -> CalibrateLeft/RightImage, BGR2HSV,
 *                                     LightingCorrection, BGR2GRAY      P/Main.cpp:351-371, 914-921
 *   usv_moving_object_distance     -> MovingObjectDistanceCalculator    P/DistanceCalculator.cpp:15-88
 *   usv_coordinate_position        -> CooridinatePositionCalculator     P/DistanceCalculator.cpp:90-141
 *   usv_pair_nearest / usv_stream_*-> CameraThread capture + timestamps P/Main.cpp:876-905
 *
 * There is NO CPU fallback behind these symbols: when no CUDA device is
 * usable `usv_create` fails with USV_ERR_NO_DEVICE and nothing else can run.
 */
#ifndef USV_B200_H
#define USV_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define USV_ABI_VERSION 5

/* ---- status codes ------------------------------------------------------ */
#define USV_OK 0
#define USV_ERR_INVALID_ARG (-1)
#define USV_ERR_CUDA (-2)
#define USV_ERR_NO_DEVICE (-3)
#define USV_ERR_UNSUPPORTED (-4)
#define USV_ERR_NOMEM (-5)

/* ---- enums (plain ints in the structs) --------------------------------- */
#define USV_COST_SAD 0  /* sum |a-b|          exact u32                       */
#define USV_COST_SSD 1  /* sum (a-b)^2        exact u32                       */
#define USV_COST_NCC 2  /* 1 - sum ab / sqrt(sum a^2 * sum b^2)        f64     */
#define USV_COST_ZNCC 3 /* 1 - zero-mean NCC from exact integer sums   f64     */
#define USV_COST_CENSUS 4 /* Hamming distance of 3x3 census bytes      exact u32   */
/* USV_COST_CENSUS. Every byte of a frame (pixel (x, y), channel c; channels are independent) becomes
 *   ct(x, y, c) = sum_{k<8} 2^k [I(n_k) < I(x, y, c)]
 * over the neighbours n_k of the same channel at (dx, dy) = (-1,-1), (0,-1), (+1,-1), (-1,0), (+1,0), (-1,+1), (0,+1),
 * (+1,+1) in that order. A neighbour outside [0, width) x [0, height) contributes bit 0; row padding is never read.
 * A window at x against a candidate at x' on row y costs
 *   H = sum_{dy<th, dx<tw, c<C} popcount(ctL(x+dx, y+dy, c) XOR ctR(x'+dx, y+dy, c))   (exact u32, at most 8 n)
 * with n = tmpl_w * tmpl_h * channels: raw_cost = H, MatchValue = H / (8 n), score unused (0). Candidates, the
 * first-minimum rule, accept test, indices, disparity, distance and the resolved map are those of the other costs.
 * The cost is unchanged by any strictly increasing intensity map applied to either frame: cameras that expose or
 * equalise each frame on its own still match. The sub-pixel entry points refuse it (USV_ERR_UNSUPPORTED). */

#define USV_DIST_NONE 0
#define USV_DIST_PINHOLE 1  /* ((201.6*4)/(disp*0.000043))/1000  P/Main.cpp:694 */
#define USV_DIST_POWERLAW 2 /* pow((10760*pow(disp,-0.877))/3.0752, 1/0.7791)
                               P/DistanceCalculator.cpp:84                    */

#define USV_LEFT_CAM 1  /* reference `#define LeftCam true`  P/DistanceCalculator.hpp:17 */
#define USV_RIGHT_CAM 0 /* reference `#define RightCam false` P/DistanceCalculator.hpp:18 */

#define USV_NO_MATCH 0xFFFFFFFFu /* RightIndex of a window with no accepted candidate */
#define USV_NO_DISPARITY 0xFFFFu
#define USV_NO_SUBPIXEL (-2147483647 - 1) /* INT32_MIN: window without a refined disparity */

/* ---- records ----------------------------------------------------------- */

/* Bit-identical to the reference's `class Match` (16 B: u32, u32, f64). */
typedef struct usv_match {
  uint32_t LeftIndex;  /* window index, row-major over the window grid        */
  uint32_t RightIndex; /* candidate index y*NXC + x' in the other frame, or
                          USV_NO_MATCH                                        */
  double MatchValue;   /* normalised cost, 0 = perfect (P/Main.cpp:400-401)   */
} usv_match;

/*
 * Search specification. Window grid: x = ix*stride_x, y = iy*stride_y for all
 * windows that fit. Candidates of the window at (x, y) lie on the same row of
 * the other frame, enumerated in ascending x' (the reference's j-minor scan,
 * P/Main.cpp:410):
 *   camera_side == LEFT : x' = x - d,  d in [search_min, search_max]
 *   camera_side == RIGHT: x' = x + d,  d in [search_min, search_max]
 * clipped to 0 <= x' <= width - tmpl_w. The first minimum in that order wins
 * (strict '>' replacement, P/Main.cpp:451). disp = d feeds the distance.
 */
typedef struct usv_search_params {
  int32_t tmpl_w, tmpl_h;
  int32_t search_min, search_max;
  int32_t stride_x, stride_y;
  int32_t cost_kind;     /* USV_COST_*  */
  int32_t camera_side;   /* USV_LEFT_CAM / USV_RIGHT_CAM */
  int32_t distance_kind; /* USV_DIST_*  */
  int32_t reserved;
  double accept_threshold; /* accept iff MatchValue < this; reference 0.75 */
} usv_search_params;

/* Frame batch layout: [n_pairs][height][row_stride] bytes, interleaved
 * channels (CV_8UC1 / CV_8UC3 style). Device-pointer entry points need the
 * base pointer and row_stride to be multiples of 16. */
typedef struct usv_frame_desc {
  int32_t width, height, channels;
  int32_t row_stride;   /* bytes between rows            */
  int64_t frame_stride; /* bytes between frames of a batch */
} usv_frame_desc;

/* Result arrays, one entry per (pair, window); any pointer may be NULL.
 * All are device pointers for *_device calls and host pointers for *_host. */
typedef struct usv_outputs {
  usv_match *matches;      /* 16-B reference records                          */
  uint32_t *right_index;   /* as usv_match.RightIndex                         */
  uint32_t *raw_cost;      /* exact integer cost of the winner (SAD/SSD/CENSUS) */
  double *score;           /* NCC / ZNCC correlation of the winner            */
  double *distance;        /* cm, f64 (reference type)                        */
  float *distance_f32;     /* cm, f32 copy for bandwidth-bound consumers      */
  uint16_t *disparity_u16; /* d of the winner or USV_NO_DISPARITY. Meant for search_min >= 0: a negative d
                            * (candidate on the other side of the window) is stored modulo 2^16, and -1 then
                            * reads as USV_NO_DISPARITY — take right_index or matches for such ranges */
  uint16_t *raw_cost_u16;  /* raw_cost as u16 (0xFFFF = no candidate): SAD or
                              CENSUS only, and only when 255*tmpl_w*tmpl_h*channels
                              (CENSUS: 8*tmpl_w*tmpl_h*channels) < 0xFFFF,
                              so that no real cost reads as "no candidate"
                              (else USV_ERR_UNSUPPORTED); lossless             */
  uint16_t *resolved_disparity_u16;
  /* Dense sweep only. The disparity map after ResolveMatchList (P/Main.cpp:432-477)
   * has run over the pair's accepted winners ON THE DEVICE: entry = d of the window's
   * winner if that record is (part of) the reference's TentativeMatch, i.e. no later
   * window of the list claims the same RightIndex with a strictly smaller MatchValue
   * (:450-451), else USV_NO_DISPARITY. With the W-entry distance table
   * (usv_distance_lut) this is what the reference exports downstream — the distance of
   * every surviving match (P/Main.cpp:1238-1259) — in 2 bytes per window. Rows of at
   * most 2048 windows. */
} usv_outputs;

/* A context owns grow-only device scratch (staging buffers, distance LUTs,
 * the workspaces of the correlation / resolve / pre-pass kernels), so calls
 * on ONE context must not overlap: one host thread at a time, and *_device
 * calls enqueued on different CUDA streams must be ordered by the caller.
 * For overlapped execution use a usv_stream (every slot owns its stream and
 * its scratch) or one context per stream; contexts are cheap. */
typedef struct usv_ctx usv_ctx;       /* one per (GPU, host thread)          */
typedef struct usv_stream usv_stream; /* pinned ring + CUDA streams          */

/* ---- lifetime ---------------------------------------------------------- */
int usv_abi_version(void);
int usv_create(int device, usv_ctx **out);
int usv_destroy(usv_ctx *ctx);
const char *usv_last_error(const usv_ctx *ctx);
/* kernels launched by this context since creation (evidence counter) */
int64_t usv_launch_count(const usv_ctx *ctx);
/* name of the kernel variant the last match call dispatched to */
const char *usv_last_kernel(const usv_ctx *ctx);
/* Per-context options. USV_OPT_CORR_KERNEL picks the sweep that serves the dense
 * NCC / ZNCC / SSD costs wherever it covers the job (a test and measurement aid:
 * the parity suite runs the same inputs through each kernel); AUTO = the
 * dispatch the library ships with. There is no environment-variable switch. */
#define USV_OPT_CORR_KERNEL 1
#define USV_CORR_KERNEL_AUTO 0
#define USV_CORR_KERNEL_ALU 1      /* IDP.4A sliding sums (usv_dense_corr.cu)    */
#define USV_CORR_KERNEL_MMA_SYNC 2 /* mma.sync IMMA      (usv_dense_mma.cu)     */
#define USV_CORR_KERNEL_TCGEN05 3  /* tcgen05 / TMEM     (usv_dense_umma.cu)    */
int usv_set_option(usv_ctx *ctx, int32_t key, int64_t value);
/* Status word the kernels of this context can raise instead of trapping (today: a
 * tcgen05 completion wait that exceeded its 10 s wall-clock bound). Returns USV_OK
 * or USV_ERR_CUDA (and clears the word). The *_host entry points and
 * usv_stream_wait check it themselves; callers of the asynchronous *_device entry
 * points check it after synchronising their stream. */
int usv_device_status(usv_ctx *ctx);

/* ---- geometry (pure host arithmetic, no device needed) ------------------ */
/* nx, ny: window grid; cand_evals: candidate evaluations per frame pair.  */
int usv_grid_dims(const usv_frame_desc *frame, const usv_search_params *params,
                  int32_t *nx, int32_t *ny, int64_t *cand_evals);

/* ---- dense sweep: every window of the grid ------------------------------ */
int usv_match_dense_device(usv_ctx *ctx, const uint8_t *d_left,
                           const uint8_t *d_right, const usv_frame_desc *frame,
                           int32_t n_pairs, const usv_search_params *params,
                           const usv_outputs *d_out, void *cuda_stream);
/* Host buffers: H2D, kernels, D2H and a final synchronise, all inside. */
int usv_match_dense_host(usv_ctx *ctx, const uint8_t *h_left,
                         const uint8_t *h_right, const usv_frame_desc *frame,
                         int32_t n_pairs, const usv_search_params *params,
                         const usv_outputs *h_out);

/* ---- sub-pixel disparity of the dense sweep's winners, 1/16 px ---------------
 * Input per window of the dense grid (layout [pair][iy*nx + ix], as usv_outputs): the RightIndex r the sweep wrote.
 * Output per window: disparity_x16 (int32, 1/16 px) and distance (f64, cm, from the refined disparity).
 *   - r == USV_NO_MATCH, or r not a candidate of its window (r / nxc != y, or x* = r % nxc outside the window's clipped
 *     candidate range): disparity_x16 = USV_NO_SUBPIXEL, distance = 0.0; no frame byte is read for it.
 *   - c(x') = the candidate's cost in the sweep's terms: SAD / SSD the exact integer cost, NCC / ZNCC MatchValue =
 *     1 - score. Refined only when x*-1 and x*+1 are both candidates of the window (in the frame and in
 *     [search_min, search_max]); otherwise q = 0.
 *   - SAD / SSD, int64: num = c(x*-1) - c(x*+1), den = c(x*-1) + c(x*+1) - 2 c(x*);
 *     den > 0: q = sgn(num) * floor((16 |num| + den) / (2 den)), clamped to [-8, 8]; else q = 0.
 *   - NCC / ZNCC, f64, every operation correctly rounded: num = v- - v+, den = (v- - v0) + (v+ - v0);
 *     den > 0: q = round(8 num / den) (half away from zero), clamped to [-8, 8]; else q = 0.
 *   - disparity_x16 = 16 d - q (USV_LEFT_CAM, d = x - x*) or 16 d + q (USV_RIGHT_CAM, d = x* - x): the parabola's
 *     vertex in 1/16 px, rounded half away from zero. distance = distance_kind's formula at disparity_x16 / 16.0.
 * For the sweep's own winners den > 0 always (the first minimum in ascending x' has c(x*-1) > c(x*) <= c(x*+1)); a tie
 * c(x*+1) == c(x*) gives q = +8, the midpoint of the tied pair. The other outputs (distance, disparity_u16, matches,
 * resolved_disparity_u16) keep the integer disparity. To combine with the resolved map, take disparity_x16 where
 * resolved_disparity_u16 != USV_NO_DISPARITY. Frames wider than 2^26 pixels are refused (USV_ERR_UNSUPPORTED), and
 * so is USV_COST_CENSUS (the pass reads frame bytes, not census bytes).
 * At least one of the two output pointers must be non-NULL. */
/* Device pointers (frames as usv_match_dense_device), enqueued on cuda_stream. */
int usv_refine_subpixel_device(usv_ctx *ctx, const uint8_t *d_left, const uint8_t *d_right,
                               const usv_frame_desc *frame, int32_t n_pairs,
                               const usv_search_params *params, const uint32_t *d_right_index,
                               int32_t *d_disparity_x16, double *d_distance, void *cuda_stream);
/* Host buffers: the dense sweep into h_out (byte for byte what usv_match_dense_host returns; h_out may be NULL or all
 * NULL, RightIndex then stays on the device), the refinement of its winners, D2H and a final synchronise.
 * usv_last_kernel names the sweep's kernel. */
int usv_match_dense_subpixel_host(usv_ctx *ctx, const uint8_t *h_left, const uint8_t *h_right,
                                  const usv_frame_desc *frame, int32_t n_pairs,
                                  const usv_search_params *params, const usv_outputs *h_out,
                                  int32_t *h_disparity_x16, double *h_distance);

/* ---- sparse templates: explicit (x, y) list, shared by all pairs -------- */
/* cost_rows (optional): [n_pairs][n_templates][row_cap] u32 costs of every
 * candidate in scan order (SAD/SSD/CENSUS); score_rows likewise f64 (NCC/ZNCC).
 * Entries past a template's candidate count are left untouched.
 * A template must fit the frame: 0 <= x <= width - tmpl_w, 0 <= y <= height -
 * tmpl_h. The *_host entry point rejects a list that violates this
 * (USV_ERR_INVALID_ARG); the *_device entry point cannot read a list that lives
 * in HBM, so its kernel writes the "no candidate" record for such a template
 * (RightIndex USV_NO_MATCH, MatchValue +inf) and touches no frame memory. */
int usv_match_templates_device(usv_ctx *ctx, const uint8_t *d_left,
                               const uint8_t *d_right,
                               const usv_frame_desc *frame, int32_t n_pairs,
                               const int32_t *d_tx, const int32_t *d_ty,
                               int32_t n_templates,
                               const usv_search_params *params,
                               const usv_outputs *d_out, uint32_t *d_cost_rows,
                               double *d_score_rows, int32_t row_cap,
                               void *cuda_stream);
int usv_match_templates_host(usv_ctx *ctx, const uint8_t *h_left,
                             const uint8_t *h_right,
                             const usv_frame_desc *frame, int32_t n_pairs,
                             const int32_t *h_tx, const int32_t *h_ty,
                             int32_t n_templates,
                             const usv_search_params *params,
                             const usv_outputs *h_out, uint32_t *h_cost_rows,
                             double *h_score_rows, int32_t row_cap);

/* ---- generate -> resolve -> distance in ONE call, host buffers: the reference's call
 * order for one frame pair (P/Main.cpp:1115-1143 then :681-694 / :1238). Dense sweep of
 * the window grid (first minimum per window, accept test :417), the reference's
 * whole-list ResolveMatchList (:432-477) over the accepted winners on the device, the
 * distance of every surviving record. h_matches / h_distance receive the first `cap`
 * records of TentativeMatch in the reference's order (duplicates and all); *n_out = its
 * full length. h_distance may be NULL. Frames go through the context's pinned staging. */
int usv_block_search_host(usv_ctx *ctx, const uint8_t *h_left,
                          const uint8_t *h_right, const usv_frame_desc *frame,
                          const usv_search_params *params, usv_match *h_matches,
                          double *h_distance, int64_t cap, int64_t *n_out);

/* ---- the reference's ORIGINAL cost: contour shape + size (P/Main.cpp:403-426) ----
 * cost(i, j) = cv::matchShapes(This[i], Other[j], CONTOURS_MATCH_I1, 0)
 *              + |area_i - area_j| / ((area_i + area_j) / 2)            (:413-415)
 * evaluated on the GPU for every pair; matches with cost < accept_threshold (:417) are written in
 * i-major / j-minor order (:408-410). Contours are concatenated (x, y) int32 pairs with CSR offsets
 * (off[k] .. off[k+1] are the points of contour k). cost_matrix (optional): all n_this * n_other
 * costs. Host pointers. */
int usv_match_contours(usv_ctx *ctx, const int32_t *pts_this,
                       const int32_t *off_this, int32_t n_this,
                       const int32_t *pts_other, const int32_t *off_other,
                       int32_t n_other, double accept_threshold,
                       usv_match *h_out, int64_t cap, int64_t *n_out,
                       double *h_cost_matrix);

/* ---- the per-frame pre-pass before the matching path, P/Main.cpp:914-921 -------------
 * camera frame (BGR, CV_8UC3) -> rectified, lighting-corrected gray frame (CV_8UC1):
 *   remap(map1 CV_16SC2, map2 CV_16UC1, INTER_LINEAR, BORDER_CONSTANT 0)   CalibrateLeft/RightImage :351-359
 *   BGR2HSV, equalizeHist(V), HSV2BGR                                      LightingCorrection :365-371, :919-920
 *   BGR2GRAY                                                               :921
 * OpenCV's arithmetic, bit for bit (oracle/preprocess_oracle.py states what is pinned against cv2 and how).
 * maps: the fixed-point pair cv::initUndistortRectifyMap(..., CV_16SC2, ...) / cv::convertMaps produce, shared
 * by all frames of the call; map1 == NULL skips the rectification. Both calls write only the width x height
 * bytes of each gray frame: row padding and the gaps between frames keep what the caller put there (a gray ROI
 * inside a larger image is safe), and the host call reads only the 3 * width x height bytes of each BGR frame. */
#define USV_PRE_OPENCV3 3 /* the reference's library: 14-bit gray coefficients, unfused HSV2BGR products */
#define USV_PRE_OPENCV4 4 /* cv2 4.13: 15-bit gray coefficients, fused `1 - s*h` (what the tests pin) */
typedef struct usv_preprocess_params {
  int32_t width, height;     /* source and destination size                         */
  int32_t src_stride;        /* bytes between BGR rows                              */
  int32_t dst_stride;        /* bytes between gray rows                             */
  int64_t src_frame_stride;  /* bytes between frames of the batch                   */
  int64_t dst_frame_stride;
  int32_t flavour;           /* USV_PRE_OPENCV3 / USV_PRE_OPENCV4                   */
  int32_t lighting;          /* 1: LightingCorrection (equalise V); 0: remap + gray */
} usv_preprocess_params;
int usv_preprocess_device(usv_ctx *ctx, const uint8_t *d_bgr, int32_t n_frames,
                          const int16_t *d_map1, const uint16_t *d_map2,
                          const usv_preprocess_params *params, uint8_t *d_gray,
                          void *cuda_stream);
int usv_preprocess_host(usv_ctx *ctx, const uint8_t *h_bgr, int32_t n_frames,
                        const int16_t *h_map1, const uint16_t *h_map2,
                        const usv_preprocess_params *params, uint8_t *h_gray);

/* ---- ResolveMatchList, P/Main.cpp:432-477, on the GPU for lists of any length ----
 * One greedy pass in list order: a match overwrites every earlier tentative entry that shares LeftIndex
 * or RightIndex (:450) and is strictly worse (:451); if it overwrote nothing it is appended (:463-466).
 * Output = the reference's TentativeMatch, duplicates and all. Returns the full output length in *n_out
 * even when it exceeds cap (only the first cap records are written).
 * skip_unmatched != 0: records with RightIndex == USV_NO_MATCH (windows without an accepted candidate,
 * as the dense kernels write them) are dropped first, as the C++ wrapper does before resolving. */
int usv_resolve_match_list(usv_ctx *ctx, const usv_match *h_in, int64_t n,
                           int32_t skip_unmatched, usv_match *h_out, int64_t cap,
                           int64_t *n_out);
/* Device pointers (d_n_out: one int64 in device memory); enqueued on cuda_stream. */
int usv_resolve_match_list_device(usv_ctx *ctx, const usv_match *d_in, int64_t n,
                                  int32_t skip_unmatched, usv_match *d_out,
                                  int64_t cap, int64_t *d_n_out, void *cuda_stream);

/* IDMatcher, P/Main.cpp:483-499: joins the current inter-frame matches with the previous ones on
 * cur.RightIndex == old.LeftIndex, i-major / j-minor. out3: (x, y, z) int32 triples; as in the reference
 * (comma operator at :492) every triple is (old.RightIndex, 0, 0). *n_out = full count even beyond cap.
 * Host pointers. */
int usv_id_matcher(usv_ctx *ctx, const usv_match *h_cur, int64_t n_cur,
                   const usv_match *h_old, int64_t n_old, int32_t *h_out3,
                   int64_t cap, int64_t *n_out);

/* ---- distance family (host buffers; one tiny kernel each) ---------------- */
/* The n-entry table distance[d], d = 0 .. n-1, built on the device by the function
 * the matching kernels' epilogue evaluates (P/Main.cpp:694 or
 * P/DistanceCalculator.cpp:84): consumers of the compact outputs (disparity_u16,
 * resolved_disparity_u16) index it instead of moving 4 or 8 more bytes per window
 * across PCIe. */
int usv_distance_lut(usv_ctx *ctx, int32_t distance_kind, int32_t n, double *h_lut);
int usv_disparity_to_distance(usv_ctx *ctx, const int32_t *h_disp, int64_t n,
                              int32_t distance_kind, double *h_dist);

/* MovingObjectDistanceCalculator, P/DistanceCalculator.cpp:15-88.
 * Points are (x, y) float pairs; idx3 is (x, y, z) int triples indexing
 * cur/old/older; timestamps are steady_clock tick counts (ns).
 * Writes n_idx distances, or nothing (returns *n_out = 0) when any of the
 * three other-camera histories is empty (:28). */
int usv_moving_object_distance(usv_ctx *ctx, int32_t camera_side,
                               int64_t t_this_ns, const float *this_xy,
                               int32_t n_this, const float *other_xy,
                               int32_t n_other, const float *old_xy,
                               int32_t n_old, const float *older_xy,
                               int32_t n_older, const int32_t *idx3,
                               int32_t n_idx, int64_t t_other_ns,
                               int64_t t_old_ns, int64_t t_older_ns,
                               double *h_dist, int32_t *n_out);

/* CooridinatePositionCalculator, P/DistanceCalculator.cpp:90-141 (without the
 * CoordinateDisplay gate, which lives in the C++ wrapper). xyz: n*3 doubles. */
int usv_coordinate_position(usv_ctx *ctx, int32_t camera_side,
                            const double *h_dist, const float *h_xy, int64_t n,
                            double *h_xyz);

/* ---- measurement aid: sustained issue rate (thread-instructions / s) of
 * VABSDIFF4.U8.ACC (which = 0) or IDP.4A.U8.U8 (which = 1) on every SM, from a
 * register-only loop timed with CUDA events for about target_ms. bench.py uses
 * it as the integer-ALU roofline denominator of the same run. */
int usv_probe_issue_rate(usv_ctx *ctx, int32_t which, double target_ms,
                         double *lane_inst_per_s);

/* ---- unsynchronized capture replacement (pure host) ---------------------- */
/* Nearest-timestamp pairing of two ascending timestamp lists (seconds):
 * each left frame takes the right frame with the smallest |tL - tR|
 * (earlier one on a tie), rejected when the gap exceeds max_dt; a right
 * frame is used at most once (the closer left frame keeps it).
 * Returns the number of pairs written (<= cap) or <0 on error. */
int64_t usv_pair_nearest(const double *t_left, int64_t n_left,
                         const double *t_right, int64_t n_right, double max_dt,
                         int32_t *out_left, int32_t *out_right, int64_t cap);

/* ---- streamed matching: pinned ring, cudaMemcpyAsync on n_slots streams -- */
#define USV_OUT_MATCHES 0x01
#define USV_OUT_RIGHT_INDEX 0x02
#define USV_OUT_RAW_COST 0x04
#define USV_OUT_SCORE 0x08
#define USV_OUT_DISTANCE 0x10
#define USV_OUT_DISTANCE_F32 0x20
#define USV_OUT_DISPARITY_U16 0x40
#define USV_OUT_RAW_COST_U16 0x80
#define USV_OUT_RESOLVED_DISPARITY_U16 0x100

int usv_stream_create(usv_ctx *ctx, const usv_frame_desc *frame,
                      const usv_search_params *params, int32_t pairs_per_slot,
                      int32_t n_slots, uint32_t output_mask, usv_stream **out);
int usv_stream_destroy(usv_stream *s);
/* Pinned staging buffers of a slot: frames laid out per `frame`, outputs
 * one entry per (pair, window). */
int usv_stream_slot(usv_stream *s, int32_t slot, uint8_t **h_left,
                    uint8_t **h_right, usv_outputs *h_out);
/* Layout of the pinned frame buffers (128-byte row pitch, packed frames). */
int usv_stream_frame_desc(const usv_stream *s, usv_frame_desc *out);
/* Enqueue H2D + kernels + D2H for the first n_pairs of the slot. */
int usv_stream_submit(usv_stream *s, int32_t slot, int32_t n_pairs);
/* Same, but the frames come from the caller's own host buffers (pinned for a
 * truly asynchronous copy) laid out per `host_frame`; results still land in the
 * slot's pinned output arrays. */
int usv_stream_submit_from(usv_stream *s, int32_t slot, const uint8_t *h_left,
                           const uint8_t *h_right,
                           const usv_frame_desc *host_frame, int32_t n_pairs);
/* Same, for unsynchronised streams (P/Main.cpp:876-905 keeps three frames per
 * camera; here the cameras write into frame stores): pair k of the slot is
 * left_store[idx_left[k]] with right_store[idx_right[k]], frames laid out per
 * `store_frame` (frame_stride = bytes between store frames), n_store_frames
 * per store. Frames go store -> HBM directly (one copy per run of consecutive
 * indices); register the stores with usv_host_register for asynchronous
 * copies. */
int usv_stream_submit_gather(usv_stream *s, int32_t slot,
                             const uint8_t *left_store, const int32_t *idx_left,
                             const uint8_t *right_store,
                             const int32_t *idx_right, int64_t n_store_frames,
                             const usv_frame_desc *store_frame,
                             int32_t n_pairs);
/* Frames from, AND results into, the caller's own host memory: every output of
 * the stream's mask is copied straight to the matching array of `h_dst` (entry 0 of
 * each array = pair 0 of this submission) instead of the slot's pinned arrays — the
 * way a multi-GPU worker lands its shard in a disjoint slice of one host result array
 * (SURVEY 8e). Page-lock both sides (usv_host_register) for asynchronous copies. */
int usv_stream_submit_io(usv_stream *s, int32_t slot, const uint8_t *h_left,
                         const uint8_t *h_right, const usv_frame_desc *host_frame,
                         int32_t n_pairs, const usv_outputs *h_dst);
/* Page-lock / release a caller-owned host buffer (frame store, result array)
 * so that copies from / to it overlap with the kernels. */
int usv_host_register(usv_ctx *ctx, void *p, size_t bytes);
int usv_host_unregister(usv_ctx *ctx, void *p);
/* Block until the slot's D2H has landed. */
int usv_stream_wait(usv_stream *s, int32_t slot);
/* Bytes moved per submitted pair (for the bench's e2e accounting). */
int usv_stream_bytes_per_pair(const usv_stream *s, int64_t *h2d, int64_t *d2h);

#ifdef __cplusplus
}
#endif
#endif /* USV_B200_H */
