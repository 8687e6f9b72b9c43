// PIL-exact antialiased bilinear resize of uint8 HWC images (SURVEY 8(f) row f1).
//
// Replaces the CPU resize inside the reference's transform (torchvision Resize -> Pillow Image.resize(BILINEAR),
// data/preprocess.py:117-121, api/inference.py:153-167).  Pillow's algorithm (src/libImaging/Resample.c, a
// third-party dependency of the reference, not vendored) is: horizontal pass first, intermediate rounded to
// uint8, then the vertical pass; each output = clip8((2^21 + sum(pixel * w)) >> 22) with 22-bit fixed-point
// triangle-filter weights.  The windows and weights come from the host (vqa_b200/resize.py computes them in
// double precision exactly like the C code); these kernels do the two integer passes, bit-exact with PIL.
// Pillow runs the vertical pass first for images more than 100 times taller than wide; the host does that as two
// single-pass calls (vqa_b200/resize.py: vertical_first).  Rows are grid-strided: gridDim.y is capped at 65 535, while
// an image may have more rows (a long screenshot).
#include "common.cuh"

namespace {

constexpr int kPrecisionBits = 32 - 8 - 2;

__device__ __forceinline__ unsigned char clip8(int v) {
  v >>= kPrecisionBits;
  return static_cast<unsigned char>(v < 0 ? 0 : (v > 255 ? 255 : v));
}

// one thread = one output pixel (all channels): dst[y, xx, :] from src[y, xmin .. xmin+n, :]
__global__ void resize_h_kernel(const unsigned char* __restrict__ src, unsigned char* __restrict__ dst, int rows, int in_w,
                                int out_w, int ch, const int* __restrict__ bounds, const int* __restrict__ kk, int ksize) {
  pdl_launch_dependents();
  pdl_wait();
  const int xx = blockIdx.x * blockDim.x + threadIdx.x;
  if (xx >= out_w) return;
  const int x0 = bounds[2 * xx], n = bounds[2 * xx + 1];
  const int* k = kk + static_cast<size_t>(xx) * ksize;
  for (int y = blockIdx.y; y < rows; y += gridDim.y) {
    const unsigned char* row = src + (static_cast<size_t>(y) * in_w + x0) * ch;
    int acc[4] = {1 << (kPrecisionBits - 1), 1 << (kPrecisionBits - 1), 1 << (kPrecisionBits - 1), 1 << (kPrecisionBits - 1)};
    for (int i = 0; i < n; ++i) {
      const int w = __ldg(k + i);
      for (int c = 0; c < ch; ++c) acc[c] += static_cast<int>(row[i * ch + c]) * w;
    }
    unsigned char* o = dst + (static_cast<size_t>(y) * out_w + xx) * ch;
    for (int c = 0; c < ch; ++c) o[c] = clip8(acc[c]);
  }
}

// one thread = one output byte column (x * ch + c) of one output row: coalesced over the row
__global__ void resize_v_kernel(const unsigned char* __restrict__ src, unsigned char* __restrict__ dst, int out_h, int row_bytes,
                                const int* __restrict__ bounds, const int* __restrict__ kk, int ksize) {
  pdl_launch_dependents();
  pdl_wait();
  const int xb = blockIdx.x * blockDim.x + threadIdx.x;
  if (xb >= row_bytes) return;
  for (int yy = blockIdx.y; yy < out_h; yy += gridDim.y) {
    const int y0 = bounds[2 * yy], n = bounds[2 * yy + 1];
    const int* k = kk + static_cast<size_t>(yy) * ksize;
    int acc = 1 << (kPrecisionBits - 1);
    for (int i = 0; i < n; ++i) acc += static_cast<int>(src[static_cast<size_t>(y0 + i) * row_bytes + xb]) * __ldg(k + i);
    dst[static_cast<size_t>(yy) * row_bytes + xb] = clip8(acc);
  }
}

constexpr int kMaxGridY = 65535;

unsigned grid_rows(int rows) { return static_cast<unsigned>(rows < kMaxGridY ? rows : kMaxGridY); }

}  // namespace

extern "C" int vqa_resize_bilinear_u8(const uint8_t* src, int32_t in_h, int32_t in_w, int32_t channels, uint8_t* tmp,
                                      uint8_t* dst, int32_t out_h, int32_t out_w, const int32_t* bounds_h,
                                      const int32_t* kk_h, int32_t ksize_h, const int32_t* bounds_v, const int32_t* kk_v,
                                      int32_t ksize_v, void* stream) {
  VQA_REQUIRE(src != nullptr && dst != nullptr, VQA_E_INVALID, "resize: null image pointer");
  VQA_REQUIRE(in_h >= 1 && in_w >= 1 && out_h >= 1 && out_w >= 1 && channels >= 1 && channels <= 4, VQA_E_INVALID,
              "resize: bad geometry (1..4 channels)");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const bool need_h = in_w != out_w, need_v = in_h != out_h;
  VQA_REQUIRE(!need_h || (bounds_h && kk_h && ksize_h >= 1), VQA_E_INVALID, "resize: missing horizontal coefficients");
  VQA_REQUIRE(!need_v || (bounds_v && kk_v && ksize_v >= 1), VQA_E_INVALID, "resize: missing vertical coefficients");
  VQA_REQUIRE(!(need_h && need_v) || tmp != nullptr, VQA_E_INVALID, "resize: two passes need the intermediate buffer");
  if (!need_h && !need_v) {
    VQA_CUDA_OK(cudaMemcpyAsync(dst, src, static_cast<size_t>(in_h) * in_w * channels, cudaMemcpyDeviceToDevice, st));
    return VQA_OK;
  }
  const uint8_t* vsrc = src;
  if (need_h) {     // horizontal pass first, over every input row (Pillow: rows the vertical pass needs = all of them)
    uint8_t* hdst = need_v ? tmp : dst;
    VQA_CUDA_OK(vqa_launch(resize_h_kernel, dim3((out_w + 127) / 128, grid_rows(in_h)), dim3(128), 0, st, src, hdst, in_h, in_w, out_w,
                           channels, bounds_h, kk_h, ksize_h));
    VQA_LAUNCH_OK("resize_h_kernel");
    vsrc = hdst;
  }
  if (need_v) {
    const int row_bytes = out_w * channels;
    VQA_CUDA_OK(vqa_launch(resize_v_kernel, dim3((row_bytes + 127) / 128, grid_rows(out_h)), dim3(128), 0, st, vsrc, dst, out_h, row_bytes,
                           bounds_v, kk_v, ksize_v));
    VQA_LAUNCH_OK("resize_v_kernel");
  }
  return VQA_OK;
}
