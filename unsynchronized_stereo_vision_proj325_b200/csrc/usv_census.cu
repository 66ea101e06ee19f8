// usv_census.cu — the 3x3 census transform of USV_COST_CENSUS (include/usv_b200.h) for sm_100a.
//
// Frames in, census frames out, in the same interleaved layout at a compact 16-byte pitch (usv_common.cuh:
// census_pitch) with the row padding zeroed. Every matching kernel then reads census frames as if they were frames:
// the SAD sweep with its Hamming arm (usv_dense_kernel.cuh), the direct form (usv_direct.cu), and the colour-plane
// split in front of the sweep. One thread makes one output word (four bytes) from three input rows, three aligned words
// a row: the neighbours of a byte lie C bytes to either side, so one funnel shift aligns a neighbour word with the
// centre word and one VSET4 (__vcmpltu4) compares four bytes at once. Memory-bound and small next to the sweep: a
// 640x480 gray pair reads and writes about 0.6 MB.
#include "usv_common.cuh"

namespace usv {

// bytes [0, n) of a word, n clamped to [0, 4]
__device__ __forceinline__ uint32_t low_bytes(int n) { return n >= 4 ? 0xffffffffu : n <= 0 ? 0u : 0xffffffffu >> (32 - 8 * n); }

// grid: (word tiles of a frame, pair of the chunk, camera)
__global__ void __launch_bounds__(256) census_transform_kernel(const DevJob J, int pair0, uint8_t* dst_l, uint8_t* dst_r, int pitch) {
  const int cam = blockIdx.z, pair = blockIdx.y;
  const int words = pitch >> 2;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= words * J.height) return;
  const int y = idx / words, w = idx - y * words;
  const uint8_t* src = (cam ? J.right : J.left) + (long long)(pair0 + pair) * J.frame_stride;
  uint32_t* dst = reinterpret_cast<uint32_t*>((cam ? dst_r : dst_l) + (long long)pair * J.height * pitch);
  const int C = J.channels, nb = J.width * C, b = 4 * w;
  uint32_t out = 0;
  if (b < nb) {
    // byte i of the word is pixel byte b + i; it has a left neighbour when b + i >= C and a right one when
    // b + i + C < nb. Words past the row are clamped onto it: what they hold is masked off.
    const uint32_t m_left = ~low_bytes(C - b), m_right = low_bytes(nb - C - b);
    const int last = (J.row_stride >> 2) - 1;
    const int s_left = 8 * (4 - C), s_right = 8 * C;  // C = 4: the neighbour word itself (shift 0 / clamped 32)
    uint32_t centre = 0;
    uint32_t nb_w[3][3];  // [row y-1, y, y+1][left, centre, right] neighbour words of the four bytes
    bool row_ok[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const int yy = y + r - 1;
      row_ok[r] = yy >= 0 && yy < J.height;
      const uint32_t* row = reinterpret_cast<const uint32_t*>(src + (long long)(row_ok[r] ? yy : y) * J.row_stride);
      const uint32_t a = __ldg(row + max(w - 1, 0)), c = __ldg(row + w), d = __ldg(row + min(w + 1, last));
      nb_w[r][0] = __funnelshift_r(a, c, s_left);
      nb_w[r][1] = c;
      nb_w[r][2] = __funnelshift_rc(c, d, s_right);
      if (r == 1) centre = c;
    }
    // bit k of a byte: neighbour k darker than the byte, neighbours in the order (dx, dy) = (-1,-1), (0,-1), (+1,-1),
    // (-1,0), (+1,0), (-1,+1), (0,+1), (+1,+1)
    const int kDx[8] = {0, 1, 2, 0, 2, 0, 1, 2}, kRow[8] = {0, 0, 0, 1, 1, 2, 2, 2};
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      if (!row_ok[kRow[k]]) continue;
      const uint32_t m = kDx[k] == 0 ? m_left : kDx[k] == 2 ? m_right : 0xffffffffu;
      out |= (__vcmpltu4(nb_w[kRow[k]][kDx[k]], centre) & m & 0x01010101u) << k;
    }
    out &= low_bytes(nb - b);  // row padding stays zero
  }
  dst[(long long)y * words + w] = out;
}

cudaError_t census_chunk(const DevJob& J, int p0, int np, uint8_t* scratch, cudaStream_t st, DevJob& Jc, int* n_launches) {
  const int pitch = census_pitch(J);
  const size_t fb = census_frame_bytes(J);
  Jc = J;
  Jc.left = scratch;
  Jc.right = scratch + np * fb;
  Jc.row_stride = pitch;
  Jc.frame_stride = (long long)fb;
  const long long words = (long long)(pitch >> 2) * J.height;
  const dim3 g((unsigned)((words + 255) / 256), np, 2);
  census_transform_kernel<<<g, 256, 0, st>>>(J, p0, scratch, scratch + np * fb, pitch);
  *n_launches += 1;
  return cudaGetLastError();
}

}  // namespace usv
