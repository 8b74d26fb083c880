// Row movers of streaming enhancement (kernels.h StreamStepDev): a step's segments are assembled from the frames
// each stream carries in its state slot plus its new frames, the mask network's output is placed in segment layout
// for the inverse STFT, and each slot then keeps what the stream's next step needs.  Pure copies: every value the
// network and the inverse STFT see is bit-identical to what the batch path computes for the whole clip.
#include "kernels.h"

namespace nhans {

namespace {

constexpr int kRowsPerBlock = 4;
constexpr int kRow = 201;

__device__ __forceinline__ float* slot_of(const StreamStepDev& p, int s) { return p.pool + (long long)p.slot[s] * p.slot_stride; }

// grid (ceil(max_rows / 4), n): segment row t of stream s <- slot row t (t < carry) or new frame t - carry
__global__ void __launch_bounds__(256) stream_assemble_kernel(const StreamStepDev p) {
  const int s = blockIdx.y;
  const long long seg0 = p.seg_offs[s];
  const int T = (int)(p.seg_offs[s + 1] - seg0), carry = p.carry[s];
  const float* slot = slot_of(p, s);
  const int t0 = blockIdx.x * kRowsPerBlock;
  for (int i = threadIdx.x; i < kRowsPerBlock * 3 * kRow; i += blockDim.x) {
    const int r = i / (3 * kRow), c = i - r * (3 * kRow), t = t0 + r;
    if (t >= T) break;
    const bool ph = c >= kRow;
    const int k = ph ? c - kRow : c;            // ph: float index within the 402 floats of a phasor row
    float v;
    if (t < carry) v = ph ? slot[kSlotPh + (long long)t * 2 * kRow + k] : slot[(long long)t * kRow + k];
    else {
      const long long nr = p.new_offs[s] + t - carry;
      v = ph ? p.new_ph[nr * 2 * kRow + k] : p.new_lm[nr * kRow + k];
    }
    if (ph) p.seg_ph[(seg0 + t) * 2 * kRow + k] = v;
    else p.seg_lm[(seg0 + t) * kRow + k] = v;
  }
  if (blockIdx.x != 0) return;
  // the denoised frames the first emitted hops overlap, in front of the row of the first window
  const int dc = p.den_carry[s];
  float* den = p.den_seg + (seg0 + p.left[s] - dc) * kRow;
  for (int i = threadIdx.x; i < dc * kRow; i += blockDim.x) den[i] = slot[kSlotDen + i];
  for (int i = threadIdx.x; i < p.n_cols; i += blockDim.x) p.cond[(long long)s * p.n_cols + i] = slot[kSlotCond + i];
}

// grid (ceil(max_wins / 4), n): window j of stream s -> den_seg row left + j
__global__ void __launch_bounds__(256) stream_den_kernel(const StreamStepDev p) {
  const int s = blockIdx.y;
  const long long w0 = p.win_offs[s];
  const int nw = (int)(p.win_offs[s + 1] - w0);
  const long long r0 = p.seg_offs[s] + p.left[s];
  const int j0 = blockIdx.x * kRowsPerBlock;
  for (int i = threadIdx.x; i < kRowsPerBlock * kRow; i += blockDim.x) {
    const int r = i / kRow, c = i - r * kRow, j = j0 + r;
    if (j >= nw) break;
    p.den_seg[(r0 + j) * kRow + c] = p.den_win[(w0 + j) * kRow + c];
  }
}

// grid (ceil(max_rows / 4), n): slot row t - keep <- segment row t (t >= keep); the last den_keep denoised frames
__global__ void __launch_bounds__(256) stream_save_kernel(const StreamStepDev p) {
  const int s = blockIdx.y;
  const long long seg0 = p.seg_offs[s];
  const int T = (int)(p.seg_offs[s + 1] - seg0), keep = p.keep[s];
  float* slot = p.pool + (long long)p.slot[s] * p.slot_stride;
  const int t0 = keep + blockIdx.x * kRowsPerBlock;
  for (int i = threadIdx.x; i < kRowsPerBlock * 3 * kRow; i += blockDim.x) {
    const int r = i / (3 * kRow), c = i - r * (3 * kRow), t = t0 + r;
    if (t >= T) break;
    if (c >= kRow) slot[kSlotPh + (long long)(t - keep) * 2 * kRow + c - kRow] = p.seg_ph[(seg0 + t) * 2 * kRow + c - kRow];
    else slot[(long long)(t - keep) * kRow + c] = p.seg_lm[(seg0 + t) * kRow + c];
  }
  if (blockIdx.x != 0) return;
  const int dk = p.den_keep[s];
  const float* den = p.den_seg + (seg0 + p.left[s] + (p.win_offs[s + 1] - p.win_offs[s]) - dk) * kRow;
  for (int i = threadIdx.x; i < dk * kRow; i += blockDim.x) slot[kSlotDen + i] = den[i];
}

}  // namespace

cudaError_t launch_stream_assemble(cudaStream_t s, const StreamStepDev& p, int max_rows) {
  if (p.n <= 0) return cudaSuccess;
  stream_assemble_kernel<<<dim3((max(max_rows, 1) + kRowsPerBlock - 1) / kRowsPerBlock, p.n), 256, 0, s>>>(p);
  return cudaGetLastError();
}

cudaError_t launch_stream_den(cudaStream_t s, const StreamStepDev& p, int max_wins) {
  if (p.n <= 0 || max_wins <= 0) return cudaSuccess;
  stream_den_kernel<<<dim3((max_wins + kRowsPerBlock - 1) / kRowsPerBlock, p.n), 256, 0, s>>>(p);
  return cudaGetLastError();
}

cudaError_t launch_stream_save(cudaStream_t s, const StreamStepDev& p, int max_rows) {
  if (p.n <= 0) return cudaSuccess;
  stream_save_kernel<<<dim3((max(max_rows, 1) + kRowsPerBlock - 1) / kRowsPerBlock, p.n), 256, 0, s>>>(p);
  return cudaGetLastError();
}

}  // namespace nhans
