// SearchAlgorithms.hpp — the search entry points of the B200 path, named and shaped after
// the reference's (P/SearchAlgorithms.hpp:28-43 declares the search family and
// ColourSearchParameters; GenerateMatchingList / ResolveMatchList are defined at
// P/Main.cpp:403-477 and declared in no header). The reference scores *contours* with
// cv::matchShapes; this path scores *pixel blocks* (SAD / SSD / NCC / ZNCC) on the GPU, so the
// contour overloads are replaced by image-view overloads with a BlockSearchSpec. Loop order
// (template-major, candidate-minor, P/Main.cpp:408-410), the accept test (`< 0.75`, :417) and
// the strict-'>' replacement rule (:451) are the reference's.
//
// The contour pre-processing family (MorphilogicalFilter, ABSDiffSearch, ColourSearch, CannySearch) is DECLARED
// at the end of this header exactly as P/SearchAlgorithms.hpp:35-43 declares it, so that a translation unit
// of the reference that names these functions compiles against this header; their bodies are OpenCV contour
// code outside the block-search path (SURVEY.md section 2) and stay with the reference's own Main.cpp.
#ifndef SearchAlgorithms_HPP
#define SearchAlgorithms_HPP

#include <vector>

#include "DistanceCalculator.hpp"
#include "Match.hpp"
#include "usv_cv_compat.hpp"

// Kept verbatim in meaning from the reference (P/SearchAlgorithms.hpp:28-33): HSV thresholds of
// the colour segmentation that used to generate candidates. Unused by the block search.
struct ColourSearchParameters {
  int iLowHue, iLowSaturation, iLowValue, iHighHue, iHighSaturation, iHighValue, iLowHue2, iHighHue2;
};

// What to score and where to look (the reference hard-codes its equivalents: accept 0.75 at
// P/Main.cpp:417, 640x480 at P/DistanceCalculator.hpp:22-23).
struct BlockSearchSpec {
  enum CostKind { SAD = 0, SSD = 1, NCC = 2, ZNCC = 3 };
  enum DistanceKind { NoDistance = 0, Pinhole = 1, PowerLaw = 2 };
  int TemplateWidth = 16, TemplateHeight = 16;
  int SearchMin = 0, SearchMax = 1 << 20;  // disparity range, clipped to the frame
  int StrideX = 1, StrideY = 1;            // window grid of the dense overload
  CostKind Cost = SAD;
  DistanceKind Distance = Pinhole;
  double AcceptThreshold = 0.75;  // accept iff MatchValue < this (P/Main.cpp:417)
  bool CameraSide = LeftCam;      // which camera ThisCamera is
  int Device = 0;                 // CUDA device of the calling thread's context
};

// The reference's own signature, unchanged (P/Main.cpp:403): contours of this camera vs contours of the
// other, cost = matchShapes(I1) + relative area difference (:413-415) evaluated on the GPU for all pairs,
// every pair with cost < 0.75 appended as {i, j, cost} in i-major / j-minor order (:408-422).
void GenerateMatchingList(std::vector<std::vector<cv::Point> > UsefulContoursL, std::vector<std::vector<cv::Point> > UsefulContoursR,
                          std::vector<Match>& Matcher);

// Dense sweep: every window of the grid over ThisCamera against its candidates on the same row
// of OtherCamera. Appends, in window order, the best ACCEPTED match of each window — what
// GenerateMatchingList followed by ResolveMatchList yields for one template's candidates
// (TentativeMatch[0], the first minimum). LeftIndex = window index (row-major), RightIndex =
// y * (width - TemplateWidth + 1) + x'. `Distances` (optional) receives the distance of each
// appended match. The caller clears the outputs, as in the reference (P/Main.cpp:842-871).
void GenerateMatchingList(const usv::ImageView& ThisCamera, const usv::ImageView& OtherCamera, const BlockSearchSpec& Spec,
                          std::vector<Match>& Matcher, std::vector<double>* Distances = nullptr);

// Explicit templates: the reference's semantics in full — EVERY candidate whose cost passes the
// accept test is appended as {i, j, cost}, i = template index (outer loop), j = candidate
// position x' (inner loop, ascending). Feed the result to ResolveMatchList.
void GenerateMatchingList(const usv::ImageView& ThisCamera, const usv::ImageView& OtherCamera,
                          std::vector<cv::Point> Templates, const BlockSearchSpec& Spec, std::vector<Match>& Matcher);

// P/Main.cpp:432-477, behaviour for behaviour (one greedy pass; a later match replaces every
// earlier tentative entry sharing Left or Right index that is strictly worse; appended when it
// replaced nothing). Used for cross-template uniqueness over the per-window winners.
void ResolveMatchList(std::vector<Match> Matcher, std::vector<Match>& TentativeMatch);

// P/Main.cpp:483-499: joins the current and the previous inter-frame match lists on
// cur.RightIndex == old.LeftIndex. Output exactly as the reference produces it: because of the comma
// operator in `(Point3i)(cur, old.RightIndex)` (:492) every triple is (old.RightIndex, 0, 0).
void IDMatcher(std::vector<Match> InterframeMatchIndexes, std::vector<Match> OldInterframeMatchIndexes,
               std::vector<cv::Point3i>& InterframeMatchIndexesComplete);

// One call per frame pair in the reference's call order (P/Main.cpp:1115-1143, then the inline
// disparity/distance of :681-694): generate -> resolve -> distance, all three on the device
// (usv_block_search_host). ExportMatches = exactly ResolveMatchList(per-window accepted winners), the
// reference's TentativeMatch entry for entry; ExportDistances[k] = distance of ExportMatches[k].
// Returns 0, or -1 on an empty frame / GPU error like the reference's thread entry points (:908-911).
int BlockSearch(bool CameraSide, const usv::ImageView* ImportGrayThisCamera, const usv::ImageView* ImportGrayOtherCamera,
                const BlockSearchSpec& Spec, std::vector<Match>& ExportMatches, std::vector<double>& ExportDistances);

// Throughput form of the same path for a BATCH of independent frame pairs on one or more GPUs of the box (SURVEY 8e,
// replacing the two free-running CameraThreads of P/Main.cpp:1407-1420 for recorded / synthetic streams): one host worker
// thread per device, each with its own context, pinned ring and CUDA streams; pair p goes to device floor(p * G / N)
// (contiguous blocks, no inter-GPU exchange); every worker lands its results in its own disjoint slice of the caller's
// arrays. Per window: ResolvedDisparity = d of the window's winner if its record survives ResolveMatchList
// (generate -> accept -> resolve all on the device), else 0xFFFF; RawCost (optional, SAD with 255 * n < 65535) = the
// winner's integer cost. Distance = DistanceTable(...)[d]. Page-lock the frame and result arrays once with
// BlockSearchPinHostBuffer for asynchronous copies (pageable memory works, slower).
struct BlockSearchBatchStats {
  double Seconds = 0.0;            // wall clock of the whole call (copies both ways included)
  int DevicesUsed = 0;
  long long PairsPerDevice[16] = {0};
};
int BlockSearchBatch(const unsigned char* LeftFrames, const unsigned char* RightFrames, int NumPairs, int Width, int Height, size_t Step,
                     size_t FrameStep, const BlockSearchSpec& Spec, const std::vector<int>& Devices, unsigned short* ResolvedDisparity,
                     unsigned short* RawCost = nullptr, BlockSearchBatchStats* Stats = nullptr);
int BlockSearchPinHostBuffer(void* Buffer, size_t Bytes, int Device = 0);
int BlockSearchUnpinHostBuffer(void* Buffer, int Device = 0);
// distance[d], d = 0 .. Count - 1, for Spec.Distance (the table the kernels' epilogue reads)
int DistanceTable(const BlockSearchSpec& Spec, int Count, std::vector<double>& Table);

// The reference's per-frame pre-pass as one GPU call (P/Main.cpp:914-921): CalibrateLeft/RightImage (:351-359,
// remap with the fixed-point maps initUndistortRectifyMap(..., CV_16SC2, ...) produces), cvtColor BGR2HSV,
// LightingCorrection (:365-371: equalizeHist on V, HSV2BGR) and cvtColor BGR2GRAY. `Map1` ([H][W][2] int16) and
// `Map2` ([H][W] uint16) may both be null (already rectified frames). `Gray` must hold Height rows of GrayStep bytes.
// OpenCV3Arithmetic = true reproduces the reference's library (14-bit gray coefficients, unfused HSV2BGR products),
// false the OpenCV 4.13 arithmetic the tests pin against cv2. Returns 0 / -1 like the reference's thread functions.
int RectifyLightingGray(const usv::ImageView& SrcBGR, const short* Map1, const unsigned short* Map2, bool Lighting,
                        unsigned char* Gray, size_t GrayStep, bool OpenCV3Arithmetic = true, int Device = 0);

// Last error text of the calling thread's GPU context ("" when none).
const char* BlockSearchLastError();

// ---- P/SearchAlgorithms.hpp:35-43, declarations kept verbatim in signature (cv:: spelled out: this header does
// not force `using namespace cv` on its includer unless DistanceCalculator.hpp's reference-compatible mode does).
// Not defined by libusv_b200: the reference compiles its own definitions (P/Main.cpp:510-721 is the CannySearch it
// actually builds). BlockSearch above is the replacement for the scoring half of CannySearch.
void MorphilogicalFilter(cv::Mat ThesholdImage);
void ABSDiffSearch(cv::Mat* Gray, cv::Mat& ThesholdImage, cv::Mat* ImportPrev, cv::Mat& ExportPrev);
void ColourSearch(cv::Mat* HSVImage, cv::Mat& ThesholdImage, ColourSearchParameters* SliderValue);
int CannySearch(bool CameraSide, cv::Mat* ImportGrayThisCamera, std::vector<std::vector<cv::Point> >* ImportCannyUsefulContoursOtherCamera,
                std::vector<cv::Point2f>* ImportVectorCenter_pointOtherCamera,
                std::vector<std::vector<cv::Point> >& ExportCannyUsefulContoursThisCamera,
                std::vector<cv::Point2f>& ExportVectorCenter_pointThisCamera, cv::Mat& ExportContourOverlay, cv::Mat& ExportDebugCannyImg);

#endif /* SearchAlgorithms_HPP */
