// Row a1 / f2: img_preprocess + padding_image (simple_romp/romp/utils.py:16-30) on the GPU:
//   cv2.cvtColor(BGR2RGB) -> centre zero-pad to a square -> cv2.resize(..., (S,S), INTER_CUBIC) -> uint8 [S,S,3]
// in ONE kernel reading the raw BGR image and writing the network's input frame.
//
// Bit-exactness target: OpenCV's own 8-bit bicubic resize (modules/imgproc/src/resize.cpp, the algorithm restated from
// its published source; pip wheels additionally carry a closed-source IPP fast path whose results differ from OpenCV's
// own code by +-1 LSB on ~3 % of the pixels and depend on the host CPU - see DESIGN 4.7):
//   * source coordinate fx = (float)((dx + 0.5) * scale - 0.5), scale = side / S in double; sx = floor(fx); fx -= sx
//   * cubic weights (A = -0.75) evaluated in fp32 in OpenCV's operation order, converted to 11-bit fixed point with
//     round-half-even (saturate_cast<short>(w * 2048)); NO renormalisation of the four taps
//   * horizontal pass in int32 over the 4 taps with replicated borders (index clamp on the padded square)
//   * vertical pass in fp32 exactly like the vectorised VResizeCubic path: t = S3*b3; t = S2*b2 + t; t = S1*b1 + t;
//     t = S0*b0 + t with b_k = beta_k * 2^-22, separate multiply and add roundings (no FMA), round-half-even, saturate.
// The zero padding and the BGR->RGB swap are folded into the tap fetch.
#include "common.cuh"

namespace b200romp {

__device__ __forceinline__ void cubic_taps(int d, double scale, int* s0, int (&w)[4]) {
  float fx = (float)(((double)d + 0.5) * scale - 0.5);
  int s = (int)fx;
  s -= (s > fx);                                   // cvFloor
  fx = __fsub_rn(fx, (float)s);
  const float A = -0.75f;
  const float x1 = __fadd_rn(fx, 1.f);
  float c0 = __fsub_rn(__fmul_rn(__fadd_rn(__fmul_rn(__fsub_rn(__fmul_rn(A, x1), __fmul_rn(5.f, A)), x1), __fmul_rn(8.f, A)), x1), __fmul_rn(4.f, A));
  float c1 = __fadd_rn(__fmul_rn(__fmul_rn(__fsub_rn(__fmul_rn(__fadd_rn(A, 2.f), fx), __fadd_rn(A, 3.f)), fx), fx), 1.f);
  const float xm = __fsub_rn(1.f, fx);
  float c2 = __fadd_rn(__fmul_rn(__fmul_rn(__fsub_rn(__fmul_rn(__fadd_rn(A, 2.f), xm), __fadd_rn(A, 3.f)), xm), xm), 1.f);
  float c3 = __fsub_rn(__fsub_rn(__fsub_rn(1.f, c0), c1), c2);
  w[0] = __float2int_rn(__fmul_rn(c0, 2048.f));
  w[1] = __float2int_rn(__fmul_rn(c1, 2048.f));
  w[2] = __float2int_rn(__fmul_rn(c2, 2048.f));
  w[3] = __float2int_rn(__fmul_rn(c3, 2048.f));
  *s0 = s;
}

// one output pixel (3 channels) of the resize of a zero-padded square of side `side`: the square holds a win_h x win_w window
// at (top, left) whose column c is image column col0 + c (columns outside 0..w-1 are zero too).  The replicated border
// applies to the padded square.
__device__ __forceinline__ void resize_pixel(const unsigned char* __restrict__ img, int h, int w, int row_stride, int win_h,
                                             int win_w, int col0, int side, int top, int left, double scale, int dx, int dy,
                                             unsigned char* __restrict__ o) {
  int sx, sy, ax[4], ay[4];
  cubic_taps(dx, scale, &sx, ax);
  cubic_taps(dy, scale, &sy, ay);
  int rows[4][3];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int py = min(max(sy + k - 1, 0), side - 1) - top;          // replicate border of the padded square, then un-pad
    int v0 = 0, v1 = 0, v2 = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int px = min(max(sx + j - 1, 0), side - 1) - left;
      const int col = col0 + px;
      if ((unsigned)py < (unsigned)win_h && (unsigned)px < (unsigned)win_w && (unsigned)col < (unsigned)w) {
        const unsigned char* p = img + (size_t)py * row_stride + (size_t)col * 3;
        v0 += (int)p[2] * ax[j];                                        // RGB <- BGR
        v1 += (int)p[1] * ax[j];
        v2 += (int)p[0] * ax[j];
      }
    }
    rows[k][0] = v0; rows[k][1] = v1; rows[k][2] = v2;
  }
  const float sc = 1.f / (2048.f * 2048.f);
  const float b0 = __fmul_rn((float)ay[0], sc), b1 = __fmul_rn((float)ay[1], sc), b2 = __fmul_rn((float)ay[2], sc), b3 = __fmul_rn((float)ay[3], sc);
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float t = __fmul_rn((float)rows[3][c], b3);
    t = __fadd_rn(__fmul_rn((float)rows[2][c], b2), t);
    t = __fadd_rn(__fmul_rn((float)rows[1][c], b1), t);
    t = __fadd_rn(__fmul_rn((float)rows[0][c], b0), t);
    o[c] = (unsigned char)min(max(__float2int_rn(t), 0), 255);
  }
}

// thread = one output pixel (3 channels)
__global__ void __launch_bounds__(256) preprocess_bgr_kernel(const unsigned char* __restrict__ img, int h, int w, int row_stride, int side,
                                                             int top, int left, double scale, int S, unsigned char* __restrict__ out) {
  const int dx = blockIdx.x * blockDim.x + threadIdx.x, dy = blockIdx.y;
  if (dx >= S) return;
  resize_pixel(img, h, w, row_stride, h, w, 0, side, top, left, scale, dx, dy, out + ((size_t)dy * S + dx) * 3);
}

// crowd mode: blockIdx.z = crop.  Crop c covers rows 0..h-1 and columns plan[c] = [l, r) of the image padded by `pad` zero
// columns on each side (split2process.py:6-39); each crop is img_preprocess'ed like a whole image (utils.py:16-30).
__global__ void __launch_bounds__(256) preprocess_crops_kernel(const unsigned char* __restrict__ img, int h, int w, int row_stride,
                                                               int pad, const int* __restrict__ plan, int first_crop, int S,
                                                               unsigned char* __restrict__ out) {
  const int dx = blockIdx.x * blockDim.x + threadIdx.x, dy = blockIdx.y, c = blockIdx.z;
  if (dx >= S) return;
  const int l = plan[2 * (first_crop + c)], r = plan[2 * (first_crop + c) + 1];
  const int cw = r - l, side = h > cw ? h : cw;
  resize_pixel(img, h, w, row_stride, h, cw, l - pad, side, (side - h) / 2, (side - cw) / 2, (double)side / (double)S, dx, dy,
               out + (((size_t)c * S + dy) * S + dx) * 3);
}

}  // namespace b200romp

using namespace b200romp;

extern "C" int b200romp_preprocess_bgr(const unsigned char* img_bgr, int h, int w, int row_stride_bytes, int out_size,
                                       unsigned char* out_rgb, float* pad_info6, b200romp_stream stream) {
  B2R_REQUIRE(img_bgr && out_rgb && h > 0 && w > 0 && row_stride_bytes >= 3 * w && out_size > 0, "preprocess_bgr: bad arguments");
  const int side = h > w ? h : w;
  const int top = (side - h) / 2, left = (side - w) / 2;
  if (pad_info6) {                     // utils.py:24: [top, bottom, left, right, h, w]
    pad_info6[0] = (float)top; pad_info6[1] = (float)(top + h); pad_info6[2] = (float)left; pad_info6[3] = (float)(left + w);
    pad_info6[4] = (float)h; pad_info6[5] = (float)w;
  }
  dim3 grid((out_size + 255) / 256, out_size);
  preprocess_bgr_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(img_bgr, h, w, row_stride_bytes, side, top, left, (double)side / (double)out_size,
                                                               out_size, out_rgb);
  B2R_CUDA_OK(cudaGetLastError());
  return B200ROMP_OK;
}

extern "C" int b200romp_preprocess_crops_bgr(const unsigned char* img_bgr, int h, int w, int row_stride_bytes, int pad,
                                             const int* plan, int first_crop, int n_crops, int out_size, unsigned char* out_rgb,
                                             b200romp_stream stream) {
  B2R_REQUIRE(img_bgr && plan && out_rgb && h > 0 && w > 0 && row_stride_bytes >= 3 * w && pad >= 0 && first_crop >= 0 &&
                  n_crops > 0 && n_crops <= 65535 && out_size > 0, "preprocess_crops_bgr: bad arguments");
  dim3 grid((out_size + 255) / 256, out_size, n_crops);
  preprocess_crops_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(img_bgr, h, w, row_stride_bytes, pad, plan, first_crop, out_size,
                                                                  out_rgb);
  B2R_CUDA_OK(cudaGetLastError());
  return B200ROMP_OK;
}
