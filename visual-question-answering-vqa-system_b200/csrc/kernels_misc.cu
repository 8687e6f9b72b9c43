// Memory-bound and small kernels of the VQA forward path (everything that is not a GEMM).
// Each launcher takes the generic VqaOp (fields in op_fields.h) with external pointers resolved.
#include <cstdlib>

#include <cuda_fp16.h>

#include "common.cuh"

namespace {

constexpr int kMaxDevices = 64;

__device__ __forceinline__ float bf16lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf16hi(uint32_t w) { return __uint_as_float(w & 0xFFFF0000u); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ------------------------------------------------------------------------------------------------
// INGEST: images -> phase-packed stem input.  Row r of the 114x114 (pad 2) grid holds the 2x2 pixel
// block (2a+ph, 2b+pw) x (R,G,B,0) as 16 bf16.  mode 0: fp32 NCHW already normalised
// (models/vqa_model.py:243-258); mode 1: uint8 HWC, normalised here exactly like
// ToTensor + Normalize (data/preprocess.py:117-121): (u8/255 - mean)/std in fp32.
// ones = 1: the two spare slots (phase (0,0) and (0,1), channel 3) of every in-image block hold 1.0 so that
// the stem GEMM adds its bias through two K columns (bias_hi + bias_lo) instead of in the epilogue.
// f32 = 1 (tf32 precision mode): the block is written as 16 tf32-rounded fp32 (64 bytes) instead of 16 bf16.
__global__ void ingest_kernel(const void* __restrict__ src, uint4* __restrict__ dst, int B, int mode, int P,
                              int rows, int ones, int f32) {
  pdl_launch_dependents();
  // uint8 mode: the 3 x 256 possible results of (u8 / 255 - mean) / std, formed once per block with the same IEEE divisions
  // ToTensor + Normalize perform (bit-exact), so a pixel costs a shared-memory lookup instead of two divisions (the kernel
  // was issue-bound on its 24 divisions and 12 byte loads per thread: 61 us per 256 images against 49 us for fp32 input)
  __shared__ float lut[3][256];
  if (mode == 1 && threadIdx.x < 256) {
    const float mean[3] = {0.485f, 0.456f, 0.406f};
    const float stdv[3] = {0.229f, 0.224f, 0.225f};
    const float f = __fdiv_rn(static_cast<float>(threadIdx.x), 255.f);
#pragma unroll
    for (int c = 0; c < 3; ++c) lut[c][threadIdx.x] = __fdiv_rn(__fsub_rn(f, mean[c]), stdv[c]);
  }
  if (mode == 1) __syncthreads();
  pdl_wait();
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  const int rpi = P * P;
  const int n = r / rpi, rem = r - n * rpi;
  const int a = rem / P, b = rem - a * P;
  uint32_t w[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  float v[2][2][4];
#pragma unroll
  for (int ph = 0; ph < 2; ++ph)
#pragma unroll
    for (int pw = 0; pw < 2; ++pw)
#pragma unroll
      for (int c = 0; c < 4; ++c) v[ph][pw][c] = 0.f;
  if (a < 112 && b < 112) {
#pragma unroll
    for (int ph = 0; ph < 2; ++ph)
#pragma unroll
      for (int pw = 0; pw < 2; ++pw) v[ph][pw][3] = (ones && ph == 0) ? 1.f : 0.f;
    if (mode == 0) {
      const float* x = reinterpret_cast<const float*>(src);
#pragma unroll
      for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int ph = 0; ph < 2; ++ph) {
          const float2 q = *reinterpret_cast<const float2*>(
              x + ((static_cast<size_t>(n) * 3 + c) * 224 + (2 * a + ph)) * 224 + 2 * b);
          v[ph][0][c] = q.x;
          v[ph][1][c] = q.y;
        }
    } else {
      const unsigned char* x = reinterpret_cast<const unsigned char*>(src);
#pragma unroll
      for (int ph = 0; ph < 2; ++ph) {
        // two pixels = 6 consecutive bytes at an even offset: three 16-bit loads
        const unsigned short* px = reinterpret_cast<const unsigned short*>(
            x + ((static_cast<size_t>(n) * 224 + (2 * a + ph)) * 224 + 2 * b) * 3);
        const uint32_t h0 = __ldg(px), h1 = __ldg(px + 1), h2 = __ldg(px + 2);
        v[ph][0][0] = lut[0][h0 & 0xFFu]; v[ph][0][1] = lut[1][h0 >> 8]; v[ph][0][2] = lut[2][h1 & 0xFFu];
        v[ph][1][0] = lut[0][h1 >> 8];    v[ph][1][1] = lut[1][h2 & 0xFFu]; v[ph][1][2] = lut[2][h2 >> 8];
      }
    }
#pragma unroll
    for (int ph = 0; ph < 2; ++ph)
#pragma unroll
      for (int pw = 0; pw < 2; ++pw) {
        w[(ph * 2 + pw) * 2 + 0] = pack_bf16x2(v[ph][pw][0], v[ph][pw][1]);
        w[(ph * 2 + pw) * 2 + 1] = pack_bf16x2(v[ph][pw][2], v[ph][pw][3]);
      }
  }
  if (f32) {
    float4* d4 = reinterpret_cast<float4*>(dst) + 4 * static_cast<size_t>(r);
#pragma unroll
    for (int ph = 0; ph < 2; ++ph)
#pragma unroll
      for (int pw = 0; pw < 2; ++pw)
        d4[ph * 2 + pw] = make_float4(round_tf32_rna(v[ph][pw][0]), round_tf32_rna(v[ph][pw][1]),
                                      round_tf32_rna(v[ph][pw][2]), round_tf32_rna(v[ph][pw][3]));
    return;
  }
  dst[2 * static_cast<size_t>(r)] = make_uint4(w[0], w[1], w[2], w[3]);
  dst[2 * static_cast<size_t>(r) + 1] = make_uint4(w[4], w[5], w[6], w[7]);
}

// MAXPOOL, fp32 grids (tf32 precision mode): one thread = one output row x 4 channels.
__global__ void maxpool_f32_kernel(const float4* __restrict__ src, float4* __restrict__ dst, int B, int C4, int Hin, int Win,
                                   int Pin, int RPIin, int Hout, int Wout, int Pout, int RPIout) {
  pdl_launch_dependents();
  pdl_wait();
  const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= static_cast<long long>(B) * RPIout * C4) return;
  const int cg = static_cast<int>(t % C4);
  const int r = static_cast<int>(t / C4);
  const int n = r / RPIout, rem = r - n * RPIout;
  const int i = rem / Pout, j = rem - i * Pout;
  float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
  if (i < Hout && j < Wout) {
    o = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    for (int dh = -1; dh <= 1; ++dh) {
      const int h = 2 * i + dh;
      if (h < 0 || h >= Hin) continue;
      for (int dw = -1; dw <= 1; ++dw) {
        const int w = 2 * j + dw;
        if (w < 0 || w >= Win) continue;
        const float4 q = src[(static_cast<size_t>(n) * RPIin + h * Pin + w) * C4 + cg];
        o.x = fmaxf(o.x, q.x); o.y = fmaxf(o.y, q.y); o.z = fmaxf(o.z, q.z); o.w = fmaxf(o.w, q.w);
      }
    }
  }
  dst[static_cast<size_t>(r) * C4 + cg] = o;
}

// ------------------------------------------------------------------------------------------------
// MAXPOOL 3x3/2 p1 on padded-flat bf16 grids; one thread = one output row x 8 channels.
__global__ void maxpool_kernel(const uint4* __restrict__ src, uint4* __restrict__ dst, int B, int C8, int Hin, int Win,
                               int Pin, int RPIin, int Hout, int Wout, int Pout, int RPIout) {
  pdl_launch_dependents();
  pdl_wait();
  const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long total = static_cast<long long>(B) * RPIout * C8;
  if (t >= total) return;
  const int cg = static_cast<int>(t % C8);
  const int r = static_cast<int>(t / C8);
  const int n = r / RPIout, rem = r - n * RPIout;
  const int i = rem / Pout, j = rem - i * Pout;
  uint4 o = make_uint4(0, 0, 0, 0);
  if (i < Hout && j < Wout) {
    __nv_bfloat162 m[4];
    bool any = false;
#pragma unroll
    for (int dh = -1; dh <= 1; ++dh) {
      const int h = 2 * i + dh;
      if (h < 0 || h >= Hin) continue;
#pragma unroll
      for (int dw = -1; dw <= 1; ++dw) {
        const int w = 2 * j + dw;
        if (w < 0 || w >= Win) continue;
        const uint4 q = src[(static_cast<size_t>(n) * RPIin + h * Pin + w) * C8 + cg];
        const __nv_bfloat162* v = reinterpret_cast<const __nv_bfloat162*>(&q);
        if (!any) {
#pragma unroll
          for (int k = 0; k < 4; ++k) m[k] = v[k];
          any = true;
        } else {
#pragma unroll
          for (int k = 0; k < 4; ++k) m[k] = __hmax2(m[k], v[k]);
        }
      }
    }
    o = *reinterpret_cast<uint4*>(m);
  }
  dst[static_cast<size_t>(r) * C8 + cg] = o;
}

// ------------------------------------------------------------------------------------------------
// SE squeeze: per-(image, channel) sum over the valid pixels of a padded-flat bf16 grid.
// grid = (B, S): every CTA reduces one slice of the image's pixels into sums[n][slice][c]; se_excite adds the
// S partials in a fixed order, so the result is deterministic (no atomics).
__global__ void se_squeeze_kernel(const uint4* __restrict__ src, float* __restrict__ sums, int C8, int H, int W, int P,
                                  int RPI) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ float red[];  // [lanes][C8*8]
  const int n = blockIdx.x;
  const int lanes = blockDim.x / C8;
  const int cg = threadIdx.x % C8, pl = threadIdx.x / C8;
  const int HW = H * W;
  const int per = (HW + gridDim.y - 1) / gridDim.y;
  const int q0 = blockIdx.y * per, q1 = min(HW, q0 + per);
  float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (pl < lanes) {
    for (int q = q0 + pl; q < q1; q += lanes) {
      const int h = q / W, w = q - h * W;
      const uint4 v = src[(static_cast<size_t>(n) * RPI + h * P + w) * C8 + cg];
      acc[0] += bf16lo(v.x); acc[1] += bf16hi(v.x); acc[2] += bf16lo(v.y); acc[3] += bf16hi(v.y);
      acc[4] += bf16lo(v.z); acc[5] += bf16hi(v.z); acc[6] += bf16lo(v.w); acc[7] += bf16hi(v.w);
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) red[(pl * C8 + cg) * 8 + k] = acc[k];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C8 * 8; c += blockDim.x) {
    float s = 0.f;
    for (int l = 0; l < lanes; ++l) s += red[l * C8 * 8 + c];
    sums[(static_cast<size_t>(n) * gridDim.y + blockIdx.y) * C8 * 8 + c] = s;
  }
}

// SE excite: scale = sigmoid(W2 relu(W1 mean)), no biases (models/attention_modules.py:84-85,116-126).
__global__ void se_excite_kernel(const float* __restrict__ sums, const float* __restrict__ w1,
                                 const float* __restrict__ w2, float* __restrict__ scale, int C, int R, int S,
                                 float inv_hw) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ float sm[];  // mean[C], hid[R]
  float* mean = sm;
  float* hid = sm + C;
  const int n = blockIdx.x;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float t = 0.f;
    for (int k = 0; k < S; ++k) t += sums[(static_cast<size_t>(n) * S + k) * C + c];   // fixed order: deterministic
    mean[c] = t * inv_hw;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  for (int r = warp; r < R; r += nw) {
    float s = 0.f;
    for (int c = lane; c < C; c += 32) s += w1[static_cast<size_t>(r) * C + c] * mean[c];
    s = warp_sum(s);
    if (lane == 0) hid[r] = fmaxf(s, 0.f);
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {   // w2 is stored transposed [R][C]: coalesced over c
    float s = 0.f;
    for (int r = 0; r < R; ++r) s += w2[static_cast<size_t>(r) * C + c] * hid[r];
    scale[static_cast<size_t>(n) * C + c] = 1.f / (1.f + expf(-s));
  }
}

// ------------------------------------------------------------------------------------------------
// Spatial attention map: channel max / mean of (x*scale), 7x7 conv over [max, avg], sigmoid.
__global__ void spatial_map_kernel(const uint4* __restrict__ src, const float* __restrict__ scale,
                                   const float* __restrict__ wconv, float* __restrict__ att, int C8, int H, int W,
                                   int P, int RPI, int ks) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ float sm[];  // mx[H*W], av[H*W], sc[C]
  const int HW = H * W, C = C8 * 8;
  float* mx = sm;
  float* av = sm + HW;
  float* sc = sm + 2 * HW;
  const int n = blockIdx.x;
  for (int c = threadIdx.x; c < C; c += blockDim.x) sc[c] = scale ? scale[static_cast<size_t>(n) * C + c] : 1.f;
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  for (int q = warp; q < HW; q += nw) {
    const int h = q / W, w = q - h * W;
    const uint4* row = src + (static_cast<size_t>(n) * RPI + h * P + w) * C8;
    float m = -INFINITY, s = 0.f;
    for (int o = lane; o < C8; o += 32) {
      const uint4 v = row[o];
      const float* k = sc + o * 8;
      const float x[8] = {bf16lo(v.x) * k[0], bf16hi(v.x) * k[1], bf16lo(v.y) * k[2], bf16hi(v.y) * k[3],
                          bf16lo(v.z) * k[4], bf16hi(v.z) * k[5], bf16lo(v.w) * k[6], bf16hi(v.w) * k[7]};
#pragma unroll
      for (int j = 0; j < 8; ++j) { m = fmaxf(m, x[j]); s += x[j]; }
    }
    m = warp_max(m);
    s = warp_sum(s);
    if (lane == 0) { mx[q] = m; av[q] = s / static_cast<float>(C); }
  }
  __syncthreads();
  const int pad = ks / 2;
  for (int q = threadIdx.x; q < HW; q += blockDim.x) {
    const int h = q / W, w = q - h * W;
    float s = 0.f;
    for (int kh = 0; kh < ks; ++kh) {
      const int hh = h + kh - pad;
      if (hh < 0 || hh >= H) continue;
      for (int kw = 0; kw < ks; ++kw) {
        const int ww = w + kw - pad;
        if (ww < 0 || ww >= W) continue;
        s += wconv[kh * ks + kw] * mx[hh * W + ww] + wconv[ks * ks + kh * ks + kw] * av[hh * W + ww];
      }
    }
    att[static_cast<size_t>(n) * HW + q] = 1.f / (1.f + expf(-s));
  }
}

// ------------------------------------------------------------------------------------------------
// STAGE_TAIL: everything between a stage's last convolution and the next stage's first one, in ONE pass
// over the feature map: SE squeeze -> excite -> (spatial attention map) -> x*scale*att -> bf16, written on
// the same grid (mode 0) or as the 4-phase split the next stage's stride-2 convolutions read (mode 1)
// (models/attention_modules.py:91-136, :198-243, :422-425; models/cnn_backbone.py:267-279).
// A cluster of CS CTAs owns one image: each CTA stages H/CS pixel rows in shared memory (the map is read
// from L2/HBM exactly once), reduces its channel sums, the cluster exchanges the CS partial sums through
// distributed shared memory (added in rank order: deterministic), every CTA runs the tiny excite MLP,
// and the scaled rows go straight from shared memory to their destination.  Spatial attention needs the
// whole image's [max, mean] maps for its 7x7 convolution and therefore runs with CS = 1 (stages 3, 4).
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ float ld_dsmem_f32(const float* local, uint32_t rank) {
  uint32_t la = static_cast<uint32_t>(__cvta_generic_to_shared(local)), ra;
  float v;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(la), "r"(rank));
  asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(ra) : "memory");
  return v;
}

constexpr int kTailThreads = 512;   // 256 measured 23 % warp occupancy and latency-bound phases (ncu, profiles/r01_g_*)

struct StageTailParams {
  const uint4* src;
  const float *w1, *w2, *wconv;
  uint4* dst;
  float *scale_out, *att_out;
  int C8, H, W, P, RPI, R, ks, mode, Po, RPIo, phase_rows, CS;
  const float* sums;   // optional: per-32-row-slab channel sums written by the producing convolution's epilogue
};

// Channel sums of image n from the slab sums of the producing GEMM (sums[s*C + c] = sum over flat rows 32s..32s+31,
// pad positions are zero there) plus, for the at most two slabs the image shares with its neighbours, the image's own
// rows read directly (bf16).  Every thread accumulates a fixed subset in a fixed order and the partial rows of
// part[] are added in index order by the caller: deterministic.  part = [parts][C] floats in shared memory.
__device__ __forceinline__ void se_slab_sums(const float* __restrict__ sums, const __nv_bfloat16* __restrict__ src, int n,
                                             int RPI, int C, float* part, int parts, int tid, int nthreads) {
  const long long r_lo = static_cast<long long>(n) * RPI, r_hi = r_lo + RPI;
  long long s_lo = (r_lo + 31) >> 5, s_hi = r_hi >> 5;
  long long head_hi = s_lo * 32, tail_lo = s_hi * 32;
  if (s_hi < s_lo) { s_hi = s_lo; head_hi = r_hi; tail_lo = r_hi; }     // the image lies inside one slab
  for (int idx = tid; idx < C * parts; idx += nthreads) {
    const int c = idx % C, pt = idx / C;
    float a = 0.f;
    for (long long sl = s_lo + pt; sl < s_hi; sl += parts) a += __ldg(sums + sl * C + c);
    for (long long r = r_lo + pt; r < head_hi; r += parts) a += __bfloat162float(src[r * C + c]);
    for (long long r = tail_lo + pt; r < r_hi; r += parts) a += __bfloat162float(src[r * C + c]);
    part[pt * C + c] = a;
  }
}

// Streaming form of the stage tail for stages WITHOUT spatial attention whose producer wrote slab sums: no staging in
// shared memory, no cluster, nothing waits on a reduction over the data -- every CTA (image n, row slice j of `split`)
// derives the image's SE scale from ~RPI/32 slab sums (a few KB from L2) and then streams its rows once:
// read 16 B, scale, write 16 B at the (phase-split) destination.  bf16 only.
constexpr int kStreamThreads = 256;
constexpr int kStreamMaxC = 512;
struct SeStreamParams {
  const uint4* src;
  uint4* dst;
  const float *sums, *w1, *w2;
  float* scale_out;
  int B, C8, H, W, P, RPI, R, mode, Po, RPIo, phase_rows, split;
};

__global__ void __launch_bounds__(kStreamThreads)
se_stream_kernel(const SeStreamParams p) {
  __shared__ float part[kStreamMaxC];      // [parts][C], parts * C <= 512
  __shared__ float mean[kStreamMaxC];
  __shared__ float sc[kStreamMaxC];
  __shared__ float hid[64];
  pdl_launch_dependents();
  pdl_wait();
  const int C8 = p.C8, C = C8 * 8, W = p.W, split = p.split;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // images in DESCENDING order: the producer wrote them ascending, so the last images are still in L2
  const int n = p.B - 1 - static_cast<int>(blockIdx.x) / split;
  const int j = static_cast<int>(blockIdx.x) % split;
  const int rows_l = p.H / split, h0 = j * rows_l;
  const int NV = rows_l * W * C8;                              // 16-byte vectors of this CTA
  const uint4* img = p.src + static_cast<size_t>(n) * p.RPI * C8;
  const int cg = tid % C8;                                     // 256 % C8 == 0: a thread keeps its channel group
  // first loads of the stream in flight while the scale is being computed
  constexpr int U = 4;
  uint4 v[U];
  auto src_of = [&](int t) -> const uint4* {
    const int q = t / C8, hl = q / W, w = q - hl * W;
    return img + (static_cast<size_t>(h0 + hl) * p.P + w) * C8 + cg;
  };
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const int t = tid + u * kStreamThreads;
    v[u] = t < NV ? __ldg(src_of(t)) : make_uint4(0u, 0u, 0u, 0u);
  }
  // ---- SE scale of image n
  const int parts = C <= kStreamMaxC / 2 ? kStreamMaxC / 2 / C * 1 : 1;   // C=64: 4, C=128: 2, C>=256: 1
  se_slab_sums(p.sums, reinterpret_cast<const __nv_bfloat16*>(p.src), n, p.RPI, C, part, parts, tid, kStreamThreads);
  __syncthreads();
  const float inv_hw = 1.f / static_cast<float>(p.H * W);
  for (int c = tid; c < C; c += kStreamThreads) {
    float t = 0.f;
    for (int l = 0; l < parts; ++l) t += part[l * C + c];
    mean[c] = t * inv_hw;
  }
  __syncthreads();
  for (int r = warp; r < p.R; r += kStreamThreads / 32) {
    float t = 0.f;
    for (int c = lane; c < C; c += 32) t += __ldg(p.w1 + static_cast<size_t>(r) * C + c) * mean[c];
    t = warp_sum(t);
    if (lane == 0) hid[r] = fmaxf(t, 0.f);
  }
  __syncthreads();
  for (int c = tid; c < C; c += kStreamThreads) {             // w2 is stored transposed [R][C]
    float t = 0.f;
    for (int r = 0; r < p.R; ++r) t += __ldg(p.w2 + static_cast<size_t>(r) * C + c) * hid[r];
    const float sg = 1.f / (1.f + expf(-t));
    sc[c] = sg;
    if (p.scale_out && j == 0) p.scale_out[static_cast<size_t>(n) * C + c] = sg;
  }
  __syncthreads();
  float k[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) k[i] = sc[cg * 8 + i];
  // ---- stream: x * scale -> bf16 at the destination (same grid, or the 4-phase split of the next stage)
  const int Po = p.Po;
  auto emit = [&](int t, const uint4& q4) {
    const int q = t / C8, hl = q / W, w = q - hl * W, h = h0 + hl;
    const uint32_t in[4] = {q4.x, q4.y, q4.z, q4.w};
    uint32_t o[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) o[i] = pack_bf16x2(bf16lo(in[i]) * k[2 * i], bf16hi(in[i]) * k[2 * i + 1]);
    size_t row;
    if (p.mode) row = static_cast<size_t>((h & 1) * 2 + (w & 1)) * p.phase_rows + static_cast<size_t>(n) * p.RPIo + (h >> 1) * Po + (w >> 1);
    else row = static_cast<size_t>(n) * p.RPIo + h * Po + w;
    p.dst[row * C8 + cg] = make_uint4(o[0], o[1], o[2], o[3]);
  };
  for (int t0 = tid; t0 < NV; t0 += U * kStreamThreads) {
    uint4 nx[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {                               // next batch in flight before this one is written
      const int t = t0 + (U + u) * kStreamThreads;
      nx[u] = t < NV ? __ldg(src_of(t)) : make_uint4(0u, 0u, 0u, 0u);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int t = t0 + u * kStreamThreads;
      if (t < NV) emit(t, v[u]);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) v[u] = nx[u];
  }
  // ---- the destination grid's zero padding that belongs to these rows
  const uint4 z = make_uint4(0u, 0u, 0u, 0u);
  const int rows_o = p.RPIo / Po;
  const int Ho = p.mode ? p.H / 2 : p.H, Wo = p.mode ? W / 2 : W, nph = p.mode ? 4 : 1;
  const int i0 = p.mode ? h0 / 2 : h0, i1 = p.mode ? (h0 + rows_l) / 2 : h0 + rows_l;
  const int padw = Po - Wo;
  for (int ph = 0; ph < nph; ++ph) {
    uint4* base = p.dst + (static_cast<size_t>(ph) * p.phase_rows + static_cast<size_t>(n) * p.RPIo) * C8;
    for (int t = tid; t < (i1 - i0) * padw * C8; t += kStreamThreads) {
      const int c = t % C8, e = t / C8, i = i0 + e / padw, jj = Wo + e % padw;
      base[(static_cast<size_t>(i) * Po + jj) * C8 + c] = z;
    }
    if (j == split - 1) {
      for (int t = tid; t < (rows_o - Ho) * Po * C8; t += kStreamThreads) base[static_cast<size_t>(Ho) * Po * C8 + t] = z;
    }
  }
}

// One group of 8 channels of one pixel: one uint4 of bf16, or (F32, the tf32 precision mode) two uint4 of fp32.
template <bool F32>
struct TailVec {
  static constexpr int N = F32 ? 2 : 1;
  uint4 q[N];
  __device__ __forceinline__ void to_float(float (&x)[8]) const {
    if constexpr (F32) {
      x[0] = __uint_as_float(q[0].x); x[1] = __uint_as_float(q[0].y); x[2] = __uint_as_float(q[0].z); x[3] = __uint_as_float(q[0].w);
      x[4] = __uint_as_float(q[1].x); x[5] = __uint_as_float(q[1].y); x[6] = __uint_as_float(q[1].z); x[7] = __uint_as_float(q[1].w);
    } else {
      x[0] = bf16lo(q[0].x); x[1] = bf16hi(q[0].x); x[2] = bf16lo(q[0].y); x[3] = bf16hi(q[0].y);
      x[4] = bf16lo(q[0].z); x[5] = bf16hi(q[0].z); x[6] = bf16lo(q[0].w); x[7] = bf16hi(q[0].w);
    }
  }
  __device__ __forceinline__ void from_float(const float (&x)[8]) {
    if constexpr (F32) {   // the next GEMM reads these as tf32 operands
      q[0] = make_uint4(__float_as_uint(round_tf32_rna(x[0])), __float_as_uint(round_tf32_rna(x[1])),
                        __float_as_uint(round_tf32_rna(x[2])), __float_as_uint(round_tf32_rna(x[3])));
      q[1] = make_uint4(__float_as_uint(round_tf32_rna(x[4])), __float_as_uint(round_tf32_rna(x[5])),
                        __float_as_uint(round_tf32_rna(x[6])), __float_as_uint(round_tf32_rna(x[7])));
    } else {
      q[0] = make_uint4(pack_bf16x2(x[0], x[1]), pack_bf16x2(x[2], x[3]), pack_bf16x2(x[4], x[5]), pack_bf16x2(x[6], x[7]));
    }
  }
  __device__ __forceinline__ void load(const uint4* base, size_t group) {
#pragma unroll
    for (int i = 0; i < N; ++i) q[i] = base[group * N + i];
  }
  __device__ __forceinline__ void store(uint4* base, size_t group) const {
#pragma unroll
    for (int i = 0; i < N; ++i) base[group * N + i] = q[i];
  }
};

// Two-pass form of the tail for SE-only stages (no spatial attention, bf16).  The staged kernel below is bound by the
// latency of its chain (load -> reduce -> cluster exchange -> excite -> apply; ncu: 26 % of the warp samples wait at a
// barrier, 2.3-2.9 TB/s at 56x56) and its ~100 KB of staged rows allow only two CTAs per SM to overlap their chains.
// Here nothing is staged: pass 1 streams the CTA's rows through registers for the channel sums, the cluster exchanges
// them, every CTA runs the excite MLP, and pass 2 reads the same rows AGAIN -- from L2, which holds the ~100 KB a CTA
// read a few microseconds earlier -- scales and writes them.  DRAM traffic stays one read + one write, but a CTA needs
// 2 KB of shared memory, so six to eight CTAs per SM (every cluster of a 256-image batch at once) overlap their chains.
// Same summation order per CTA as the staged kernel's 256-thread form; images are independent (batch-invariant).
constexpr int kTwoPassThreads = 256;   // four CTAs per SM; 128-thread CTAs (eight per SM) measured 64 -> 68 us at 56x56
__global__ void __launch_bounds__(kTwoPassThreads, 4)
se_two_pass_kernel(const StageTailParams p) {
  __shared__ float red[2048];             // [part_rows][C]: 8 x 64, 8 x 128, 8 x 256 or 4 x 512
  __shared__ float part[512], mean[512], sc[512], hid[64];
  pdl_launch_dependents();
  pdl_wait();
  const int C8 = p.C8, C = C8 * 8, W = p.W, CS = p.CS, R = p.R;
  const int rows_l = p.H / CS;
  const int n = static_cast<int>(gridDim.x / CS) - 1 - static_cast<int>(blockIdx.x) / CS;   // descending: the last images are still in L2
  const int rank = CS > 1 ? static_cast<int>(cluster_ctarank()) : 0;
  const int h0 = rank * rows_l;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int lanes = kTwoPassThreads / C8;
  const int cg = tid % C8, pl = tid / C8;
  const int lpw = C8 < 32 ? 32 / C8 : 1;
  const int part_rows = lanes / lpw;
  const uint4* img = p.src + static_cast<size_t>(n) * p.RPI * C8;
  // ---- pass 1: channel sums.  The CTA's rows are ONE contiguous run of rows_l * P pixels when the pad pixel that ends
  // every grid row is included; pads are zero by the layout's invariant (every producer masks them), so they add nothing.
  // Thread t walks vectors t, t + T, ... of that run: T is a multiple of C8, so its channel group never changes and the
  // loop is a load, 16 unpack / add instructions and a pointer bump (the kernel is issue-bound, not bandwidth-bound:
  // ncu showed 150 warp instructions per 16-byte vector over the two passes of the first version).
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  {
    const uint4* run = img + static_cast<size_t>(h0) * p.P * C8;
    const int NV = rows_l * p.P * C8;
    constexpr int U = 8;
    int v = tid;
    for (; v + (U - 1) * kTwoPassThreads < NV; v += U * kTwoPassThreads) {
      uint4 x[U];
#pragma unroll
      for (int u = 0; u < U; ++u) x[u] = __ldg(run + v + u * kTwoPassThreads);
#pragma unroll
      for (int u = 0; u < U; ++u) {
        acc[0] += bf16lo(x[u].x); acc[1] += bf16hi(x[u].x); acc[2] += bf16lo(x[u].y); acc[3] += bf16hi(x[u].y);
        acc[4] += bf16lo(x[u].z); acc[5] += bf16hi(x[u].z); acc[6] += bf16lo(x[u].w); acc[7] += bf16hi(x[u].w);
      }
    }
    for (; v < NV; v += kTwoPassThreads) {
      const uint4 x = __ldg(run + v);
      acc[0] += bf16lo(x.x); acc[1] += bf16hi(x.x); acc[2] += bf16lo(x.y); acc[3] += bf16hi(x.y);
      acc[4] += bf16lo(x.z); acc[5] += bf16hi(x.z); acc[6] += bf16lo(x.w); acc[7] += bf16hi(x.w);
    }
  }
  for (int off = C8; off < 32; off <<= 1) {             // C8 < 32: the warp's pixel lanes first (fixed order)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], off);
  }
  if (pl % lpw == 0) {
    const int prow = pl / lpw;
#pragma unroll
    for (int j = 0; j < 8; ++j) red[prow * C + cg * 8 + j] = acc[j];
  }
  __syncthreads();
  for (int c = tid; c < C; c += kTwoPassThreads) {
    float t = 0.f;
    for (int l = 0; l < part_rows; ++l) t += red[l * C + c];
    part[c] = t;
  }
  if (CS > 1) cluster_sync_all(); else __syncthreads();
  const float inv_hw = 1.f / static_cast<float>(p.H * W);
  for (int c = tid; c < C; c += kTwoPassThreads) {
    float t = 0.f;
    if (CS > 1) {
      for (int r = 0; r < CS; ++r) t += ld_dsmem_f32(part + c, static_cast<uint32_t>(r));
    } else {
      t = part[c];
    }
    mean[c] = t * inv_hw;
  }
  __syncthreads();
  // ---- excite: one warp per hidden unit, then one thread per channel
  for (int r = warp; r < R; r += kTwoPassThreads / 32) {
    float t = 0.f;
    for (int c = lane; c < C; c += 32) t += __ldg(p.w1 + static_cast<size_t>(r) * C + c) * mean[c];
    t = warp_sum(t);
    if (lane == 0) hid[r] = fmaxf(t, 0.f);
  }
  __syncthreads();
  for (int c = tid; c < C; c += kTwoPassThreads) {      // w2 is stored transposed [R][C]
    float t = 0.f;
    for (int r = 0; r < R; ++r) t += __ldg(p.w2 + static_cast<size_t>(r) * C + c) * hid[r];
    const float sg = 1.f / (1.f + expf(-t));
    sc[c] = sg;
    if (p.scale_out && rank == 0) p.scale_out[static_cast<size_t>(n) * C + c] = sg;
  }
  __syncthreads();
  // ---- pass 2: the same rows again (L2), scaled, to the destination grid.  A thread keeps its pixel column w and walks
  // down the rows four at a time: the source advances by one grid row, the destination alternates between the two
  // phases of the row parity (mode 1: rows come in even / odd pairs because h0 and rows_l are even) -- pointer bumps only.
  float kk[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) kk[j] = sc[cg * 8 + j];
  const int Po = p.Po;
  auto scaled = [&](const uint4& x) {
    return make_uint4(pack_bf16x2(bf16lo(x.x) * kk[0], bf16hi(x.x) * kk[1]), pack_bf16x2(bf16lo(x.y) * kk[2], bf16hi(x.y) * kk[3]),
                      pack_bf16x2(bf16lo(x.z) * kk[4], bf16hi(x.z) * kk[5]), pack_bf16x2(bf16lo(x.w) * kk[6], bf16hi(x.w) * kk[7]));
  };
  const size_t srow = static_cast<size_t>(p.P) * C8;            // source vectors per grid row
  for (int w = pl; w < W; w += lanes) {
    const uint4* s = img + (static_cast<size_t>(h0) * p.P + w) * C8 + cg;
    if (p.mode) {
      // even rows -> phase (0, w & 1), odd rows -> phase (1, w & 1); both at position (h >> 1, w >> 1)
      uint4* dE = p.dst + (static_cast<size_t>(w & 1) * p.phase_rows + static_cast<size_t>(n) * p.RPIo +
                           static_cast<size_t>(h0 >> 1) * Po + (w >> 1)) * C8 + cg;
      uint4* dO = dE + 2 * static_cast<size_t>(p.phase_rows) * C8;
      const size_t dstep = static_cast<size_t>(Po) * C8;
      int hl = 0;
      for (; hl + 4 <= rows_l; hl += 4) {
        const uint4 x0 = __ldg(s), x1 = __ldg(s + srow), x2 = __ldg(s + 2 * srow), x3 = __ldg(s + 3 * srow);
        dE[0] = scaled(x0); dO[0] = scaled(x1); dE[dstep] = scaled(x2); dO[dstep] = scaled(x3);
        s += 4 * srow; dE += 2 * dstep; dO += 2 * dstep;
      }
      for (; hl < rows_l; hl += 2) {
        const uint4 x0 = __ldg(s), x1 = __ldg(s + srow);
        dE[0] = scaled(x0); dO[0] = scaled(x1);
        s += 2 * srow; dE += dstep; dO += dstep;
      }
    } else {
      uint4* d = p.dst + (static_cast<size_t>(n) * p.RPIo + static_cast<size_t>(h0) * Po + w) * C8 + cg;
      const size_t dstep = static_cast<size_t>(Po) * C8;
      int hl = 0;
      for (; hl + 4 <= rows_l; hl += 4) {
        const uint4 x0 = __ldg(s), x1 = __ldg(s + srow), x2 = __ldg(s + 2 * srow), x3 = __ldg(s + 3 * srow);
        d[0] = scaled(x0); d[dstep] = scaled(x1); d[2 * dstep] = scaled(x2); d[3 * dstep] = scaled(x3);
        s += 4 * srow; d += 4 * dstep;
      }
      for (; hl < rows_l; ++hl) {
        d[0] = scaled(__ldg(s));
        s += srow; d += dstep;
      }
    }
  }
  // ---- the destination grid's zero padding that belongs to these rows
  const uint4 z = make_uint4(0u, 0u, 0u, 0u);
  const int rows_o = p.RPIo / Po;
  const int Ho = p.mode ? p.H / 2 : p.H, Wo = p.mode ? W / 2 : W, nph = p.mode ? 4 : 1;
  const int i0 = p.mode ? h0 / 2 : h0, i1 = p.mode ? (h0 + rows_l) / 2 : h0 + rows_l;
  const int padw = Po - Wo;
  for (int ph = 0; ph < nph; ++ph) {
    uint4* base = p.dst + (static_cast<size_t>(ph) * p.phase_rows + static_cast<size_t>(n) * p.RPIo) * C8;
    for (int t = tid; t < (i1 - i0) * padw * C8; t += kTwoPassThreads) {
      const int c = t % C8, e = t / C8, i = i0 + e / padw, j = Wo + e % padw;
      base[(static_cast<size_t>(i) * Po + j) * C8 + c] = z;
    }
    if (rank == CS - 1) {
      for (int t = tid; t < (rows_o - Ho) * Po * C8; t += kTwoPassThreads) base[static_cast<size_t>(Ho) * Po * C8 + t] = z;
    }
  }
  if (CS > 1) cluster_sync_all();                       // peers may still be reading this CTA's partial sums
}

template <bool F32>
__global__ void __launch_bounds__(kTailThreads)
stage_tail_kernel(const StageTailParams p) {
  using Vec = TailVec<F32>;
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ __align__(16) uint8_t tail_smem[];
  const int C8 = p.C8, C = C8 * 8, W = p.W, CS = p.CS;
  const int rows_l = p.H / CS;                          // pixel rows of this CTA
  const int NP = rows_l * W;                            // pixels of this CTA
  // images in DESCENDING order: the producer (conv2) wrote them ascending, so the last images are still in L2
  const int n = static_cast<int>(gridDim.x / CS) - 1 - static_cast<int>(blockIdx.x) / CS;
  const int rank = CS > 1 ? static_cast<int>(cluster_ctarank()) : 0;
  const int h0 = rank * rows_l;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int lanes = kTailThreads / C8;                  // pixel lanes (C8 divides 256)
  const int cg = tid % C8, pl = tid / C8;
  uint4* tile = reinterpret_cast<uint4*>(tail_smem);                       // [NP][C8] groups of 8 channels
  const int lpw = C8 < 32 ? 32 / C8 : 1;                // pixel lanes that share one warp (reduced by shuffles)
  const int part_rows = lanes / lpw;                    // partial sums left after the in-warp reduction
  const int red_rows = part_rows > 8 ? part_rows / 2 : part_rows;   // rows of the shared-memory scratch (folded once if > 8)
  float* red = reinterpret_cast<float*>(tile + static_cast<size_t>(NP) * C8 * Vec::N);   // [red_rows][C]; later mx/av maps
  float* part = red + red_rows * C;                     // [C] this CTA's channel sums (read by the cluster)
  float* sc = part + C;                                 // [C] SE scale
  float* hid = sc + C;                                  // [R]
  float* att = hid + 256;                               // [NP] spatial attention (CS == 1)
  float* wc = att + NP;                                 // [2*ks*ks] spatial conv weights
  const bool use_se = p.w1 != nullptr;

  // ---- 1. stage the rows with cp.async (every 16-byte piece of the CTA's rows in flight at once: one DRAM round
  // trip instead of a register-limited sequence of them), then accumulate the channel sums from shared memory
  const uint4* img = p.src + static_cast<size_t>(n) * p.RPI * C8 * Vec::N;
  // pixel q = pl, pl + lanes, ...: (row, column) are kept incrementally (ncu: the two q / W divisions of this kernel were
  // 12 % of its instructions, and the kernel is issue-bound)
  const int dq_h = lanes / W, dq_w = lanes - dq_h * W;
  int hl_s = pl / W, w_s = pl - hl_s * W;
  for (int q = pl; q < NP; q += lanes) {
    const int hl = hl_s, w = w_s;
    hl_s += dq_h; w_s += dq_w;
    if (w_s >= W) { w_s -= W; ++hl_s; }
    const uint4* g = img + ((static_cast<size_t>(h0 + hl) * p.P + w) * C8 + cg) * Vec::N;
    uint4* d = tile + (static_cast<size_t>(q) * C8 + cg) * Vec::N;
#pragma unroll
    for (int i = 0; i < Vec::N; ++i)
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(static_cast<uint32_t>(__cvta_generic_to_shared(d + i))),
                   "l"(g + i) : "memory");
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
  const bool slab = use_se && p.sums != nullptr && !F32 && CS == 1;   // channel sums come from the producer's epilogue
  if (slab) {   // (while the rows are in flight)
    const int parts = red_rows < 4 ? red_rows : 4;
    se_slab_sums(p.sums, reinterpret_cast<const __nv_bfloat16*>(p.src), n, p.RPI, C, red, parts, tid, kTailThreads);
    __syncthreads();
    for (int c = tid; c < C; c += kTailThreads) {
      float t = 0.f;
      for (int l = 0; l < parts; ++l) t += red[l * C + c];
      part[c] = t;
    }
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (use_se && !slab) {
    for (int q = pl; q < NP; q += lanes) {
      Vec v;
      v.load(tile, static_cast<size_t>(q) * C8 + cg);
      float x[8];
      v.to_float(x);
#pragma unroll
      for (int k = 0; k < 8; ++k) acc[k] += x[k];
    }
  }
  if (use_se && !slab) {
    for (int off = C8; off < 32; off <<= 1) {           // C8 < 32: the warp's pixel lanes first (fixed order)
#pragma unroll
      for (int k = 0; k < 8; ++k) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], off);
    }
    const int prow = pl / lpw;
    if (part_rows > 8) {                                // fold the upper half of the partial rows onto the lower half
      if (pl % lpw == 0 && prow >= red_rows) {
#pragma unroll
        for (int k = 0; k < 8; ++k) red[(prow - red_rows) * C + cg * 8 + k] = acc[k];
      }
      __syncthreads();
      if (pl % lpw == 0 && prow < red_rows) {
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[k] += red[prow * C + cg * 8 + k];
      }
      __syncthreads();
    }
    if (pl % lpw == 0 && prow < red_rows) {
#pragma unroll
      for (int k = 0; k < 8; ++k) red[prow * C + cg * 8 + k] = acc[k];
    }
    __syncthreads();
    for (int c = tid; c < C; c += kTailThreads) {
      float t = 0.f;
      for (int l = 0; l < red_rows; ++l) t += red[l * C + c];
      part[c] = t;
    }
  }
  if (use_se) {
    // ---- 2. cluster-wide channel sums (rank order) -> mean
    if (CS > 1) cluster_sync_all(); else __syncthreads();
    const float inv_hw = 1.f / static_cast<float>(p.H * W);
    float* mean = red;                                  // red is free again
    for (int c = tid; c < C; c += kTailThreads) {
      float t = 0.f;
      if (CS > 1) {
        for (int r = 0; r < CS; ++r) t += ld_dsmem_f32(part + c, static_cast<uint32_t>(r));
      } else {
        t = part[c];
      }
      mean[c] = t * inv_hw;
    }
    __syncthreads();
    // ---- 3. excite: scale = sigmoid(W2 relu(W1 mean)), no biases
    // 8 lanes per hidden unit, every lane's loads independent (one L2 round trip instead of a chain)
    for (int r0 = 0; r0 < p.R; r0 += kTailThreads / 8) {
      const int r = r0 + (tid >> 3), part8 = tid & 7;
      float t = 0.f;
      if (r < p.R) {
        const float4* wrow = reinterpret_cast<const float4*>(p.w1 + static_cast<size_t>(r) * C);
#pragma unroll 4
        for (int c4 = part8; c4 < C / 4; c4 += 8) {
          const float4 wv = __ldg(wrow + c4);
          const float4 mv = *reinterpret_cast<const float4*>(mean + 4 * c4);
          t += wv.x * mv.x + wv.y * mv.y + wv.z * mv.z + wv.w * mv.w;
        }
      }
      t += __shfl_xor_sync(0xffffffffu, t, 1);
      t += __shfl_xor_sync(0xffffffffu, t, 2);
      t += __shfl_xor_sync(0xffffffffu, t, 4);
      if (r < p.R && part8 == 0) hid[r] = fmaxf(t, 0.f);
    }
    __syncthreads();
    for (int c = tid; c < C; c += kTailThreads) {       // w2 is stored transposed [R][C]: coalesced over c
      float t = 0.f;
#pragma unroll 8
      for (int r = 0; r < p.R; ++r) t += __ldg(p.w2 + static_cast<size_t>(r) * C + c) * hid[r];
      const float sg = 1.f / (1.f + expf(-t));
      sc[c] = sg;
      if (p.scale_out && rank == 0) p.scale_out[static_cast<size_t>(n) * C + c] = sg;
    }
  } else {
    for (int c = tid; c < C; c += kTailThreads) sc[c] = 1.f;
  }
  __syncthreads();

  // ---- 4. spatial attention (CS == 1): channel max / mean of x*scale, ks x ks conv over [max, avg], sigmoid
  const bool use_sp = p.wconv != nullptr;
  if (use_sp) {
    float* mx = red;                                    // [NP]
    float* av = red + NP;                               // [NP]  (2*NP <= lanes*C floats, checked on the host)
    // one warp reduces 4 pixels at a time: the 4 x (max, sum) shuffle trees are independent and pipeline
    for (int q0 = warp * 4; q0 < NP; q0 += (kTailThreads / 32) * 4) {
      float m[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY}, t[4] = {0.f, 0.f, 0.f, 0.f};
      for (int o = lane; o < C8; o += 32) {
        const float* k = sc + o * 8;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (q0 + u < NP) {
            Vec v;
            v.load(tile, static_cast<size_t>(q0 + u) * C8 + o);
            float x[8];
            v.to_float(x);
#pragma unroll
            for (int j = 0; j < 8; ++j) { const float y = x[j] * k[j]; m[u] = fmaxf(m[u], y); t[u] += y; }
          }
        }
      }
#pragma unroll
      for (int sh = 16; sh > 0; sh >>= 1) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          m[u] = fmaxf(m[u], __shfl_xor_sync(0xffffffffu, m[u], sh));
          t[u] += __shfl_xor_sync(0xffffffffu, t[u], sh);
        }
      }
      if (lane < 4 && q0 + lane < NP) {
        const float mm = lane == 0 ? m[0] : lane == 1 ? m[1] : lane == 2 ? m[2] : m[3];
        const float tt = lane == 0 ? t[0] : lane == 1 ? t[1] : lane == 2 ? t[2] : t[3];
        mx[q0 + lane] = mm;
        av[q0 + lane] = tt / static_cast<float>(C);
      }
    }
    const int ks = p.ks, pad = ks / 2, H = p.H;
    for (int t = tid; t < 2 * ks * ks; t += kTailThreads) wc[t] = __ldg(p.wconv + t);
    __syncthreads();
    for (int q = tid; q < NP; q += kTailThreads) {
      const int h = q / W, w = q - h * W;
      float t = 0.f;
      for (int kh = 0; kh < ks; ++kh) {
        const int hh = h + kh - pad;
        if (hh < 0 || hh >= H) continue;
        for (int kw = 0; kw < ks; ++kw) {
          const int ww = w + kw - pad;
          if (ww < 0 || ww >= W) continue;
          t += wc[kh * ks + kw] * mx[hh * W + ww] + wc[ks * ks + kh * ks + kw] * av[hh * W + ww];
        }
      }
      const float a = 1.f / (1.f + expf(-t));
      att[q] = a;
      if (p.att_out) p.att_out[static_cast<size_t>(n) * NP + q] = a;
    }
    __syncthreads();
  }

  // ---- 5. apply and write (plus the destination grid's zero padding that belongs to these rows)
  float k[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) k[j] = sc[cg * 8 + j];
  const int Po = p.Po;
  const int rows_o = p.RPIo / Po;                       // destination rows per image incl. padding
  int hl_a = pl / W, w_a = pl - hl_a * W;
  for (int q = pl; q < NP; q += lanes) {
    const int w = w_a, h = h0 + hl_a;
    hl_a += dq_h; w_a += dq_w;
    if (w_a >= W) { w_a -= W; ++hl_a; }
    Vec v, o;
    v.load(tile, static_cast<size_t>(q) * C8 + cg);
    const float a = use_sp ? att[q] : 1.f;
    float x[8];
    v.to_float(x);
#pragma unroll
    for (int j = 0; j < 8; ++j) x[j] = x[j] * k[j] * a;
    o.from_float(x);
    size_t row;
    if (p.mode) row = static_cast<size_t>((h & 1) * 2 + (w & 1)) * p.phase_rows + static_cast<size_t>(n) * p.RPIo + (h >> 1) * Po + (w >> 1);
    else row = static_cast<size_t>(n) * p.RPIo + h * Po + w;
    o.store(p.dst, row * C8 + cg);
  }
  const uint4 z = make_uint4(0u, 0u, 0u, 0u);
  const int Ho = p.mode ? p.H / 2 : p.H, Wo = p.mode ? W / 2 : W, nph = p.mode ? 4 : 1;
  const int i0 = p.mode ? h0 / 2 : h0, i1 = p.mode ? (h0 + rows_l) / 2 : h0 + rows_l;
  const int padw = Po - Wo;                             // pad columns per destination row
  for (int ph = 0; ph < nph; ++ph) {
    constexpr int VN = Vec::N;
    const int CV = C8 * VN;                                                  // 16-byte vectors per pixel
    uint4* base = p.dst + (static_cast<size_t>(ph) * p.phase_rows + static_cast<size_t>(n) * p.RPIo) * CV;
    for (int t = tid; t < (i1 - i0) * padw * CV; t += kTailThreads) {      // pad columns of this CTA's rows
      const int c = t % CV, e = t / CV, i = i0 + e / padw, j = Wo + e % padw;
      base[(static_cast<size_t>(i) * Po + j) * CV + c] = z;
    }
    if (rank == CS - 1) {                                                   // pad rows below the image
      for (int t = tid; t < (rows_o - Ho) * Po * CV; t += kTailThreads) base[static_cast<size_t>(Ho) * Po * CV + t] = z;
    }
  }
  if (CS > 1) cluster_sync_all();                       // peers may still be reading this CTA's partial sums
}

// ------------------------------------------------------------------------------------------------
// SPLIT_TF32 (tf32 precision mode): dst[m, 0:K] = tf32(src[m, :]), dst[m, K:2K] = tf32(src - hi): the A operand
// of a 3xTF32 GEMM (program.py::linear).  One thread = 4 columns.
__global__ void split_tf32_kernel(const float* __restrict__ src, float* __restrict__ dst, int M, int K4, int ld_src) {
  pdl_launch_dependents();
  pdl_wait();
  const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= static_cast<long long>(M) * K4) return;
  const int m = static_cast<int>(t / K4), c4 = static_cast<int>(t - static_cast<long long>(m) * K4);
  const float4 x = *reinterpret_cast<const float4*>(src + static_cast<size_t>(m) * ld_src + 4 * c4);
  const float4 hi = make_float4(round_tf32_rna(x.x), round_tf32_rna(x.y), round_tf32_rna(x.z), round_tf32_rna(x.w));
  const float4 lo = make_float4(round_tf32_rna(x.x - hi.x), round_tf32_rna(x.y - hi.y), round_tf32_rna(x.z - hi.z),
                                round_tf32_rna(x.w - hi.w));
  float* drow = dst + static_cast<size_t>(m) * 8 * K4;
  *reinterpret_cast<float4*>(drow + 4 * c4) = hi;
  *reinterpret_cast<float4*>(drow + 4 * K4 + 4 * c4) = lo;
}

// ------------------------------------------------------------------------------------------------
// COPY_ROWS: dst[r, c] = src[r, c] between two leading dimensions (un-padding of the logits).
__global__ void copy_rows_kernel(const float* __restrict__ src, float* __restrict__ dst, int rows, int cols, int ld_src,
                                 int ld_dst) {
  pdl_launch_dependents();
  pdl_wait();
  const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= static_cast<long long>(rows) * cols) return;
  const int r = static_cast<int>(t / cols), c = static_cast<int>(t - static_cast<long long>(r) * cols);
  dst[static_cast<size_t>(r) * ld_dst + c] = src[static_cast<size_t>(r) * ld_src + c];
}

// ------------------------------------------------------------------------------------------------
// x*scale[c]*att[pixel] -> bf16, written either on the same grid (mode 0) or as the 4-phase split
// the next stage's stride-2 convolutions read (mode 1).  One thread = one dst row x 8 channels.
__global__ void scale_relayout_kernel(const uint4* __restrict__ src, const float* __restrict__ scale,
                                      const float* __restrict__ att, uint4* __restrict__ dst, int B, int C8, int H,
                                      int W, int P, int RPI, int mode, int Po, int RPIo, int phase_rows) {
  pdl_launch_dependents();
  pdl_wait();
  const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long total_rows = mode ? 4LL * phase_rows : static_cast<long long>(B) * RPIo;
  if (t >= total_rows * C8) return;
  const int cg = static_cast<int>(t % C8);
  const long long r = t / C8;
  int ph = 0, pw = 0;
  long long rr = r;
  if (mode) {
    const int phase = static_cast<int>(r / phase_rows);
    rr = r - static_cast<long long>(phase) * phase_rows;
    ph = phase >> 1;
    pw = phase & 1;
  }
  const int n = static_cast<int>(rr / RPIo), rem = static_cast<int>(rr - static_cast<long long>(n) * RPIo);
  const int i = rem / Po, j = rem - i * Po;
  const int Ho = mode ? H / 2 : H, Wo = mode ? W / 2 : W;
  uint4 o = make_uint4(0, 0, 0, 0);
  if (i < Ho && j < Wo) {
    const int h = mode ? 2 * i + ph : i, w = mode ? 2 * j + pw : j;
    const uint4 v = src[(static_cast<size_t>(n) * RPI + h * P + w) * C8 + cg];
    const float a = att ? att[static_cast<size_t>(n) * H * W + h * W + w] : 1.f;
    float k[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) k[q] = scale ? scale[static_cast<size_t>(n) * C8 * 8 + cg * 8 + q] : 1.f;
    o.x = pack_bf16x2(bf16lo(v.x) * k[0] * a, bf16hi(v.x) * k[1] * a);
    o.y = pack_bf16x2(bf16lo(v.y) * k[2] * a, bf16hi(v.y) * k[3] * a);
    o.z = pack_bf16x2(bf16lo(v.z) * k[4] * a, bf16hi(v.z) * k[5] * a);
    o.w = pack_bf16x2(bf16lo(v.w) * k[6] * a, bf16hi(v.w) * k[7] * a);
  }
  dst[static_cast<size_t>(r) * C8 + cg] = o;
}

__global__ void grid_to_nchw_kernel(const void* __restrict__ src_, float* __restrict__ dst, int B, int C,
                                    int H, int W, int P, int RPI, int f32) {
  pdl_launch_dependents();
  pdl_wait();
  const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= static_cast<long long>(B) * C * H * W) return;
  const int w = static_cast<int>(t % W);
  const int h = static_cast<int>((t / W) % H);
  const int c = static_cast<int>((t / (static_cast<long long>(W) * H)) % C);
  const int n = static_cast<int>(t / (static_cast<long long>(W) * H * C));
  const size_t at = (static_cast<size_t>(n) * RPI + h * P + w) * C + c;
  dst[t] = f32 ? reinterpret_cast<const float*>(src_)[at] : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(src_)[at]);
}

// ------------------------------------------------------------------------------------------------
// attention_mask (int64 | fp32 | int32 | uint8 / bool) -> binary int32 key mask of the self-attention (mask == 0 -> -inf,
// models/text_encoder.py:244) and fp32 pooling weights attention_mask.float() (models/fusion.py:299-312)
__global__ void mask_prep_kernel(const void* __restrict__ src, int* __restrict__ dst, float* __restrict__ dstf, int n,
                                 int dtype) {
  pdl_launch_dependents();
  pdl_wait();
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  float v = 1.f;
  if (dtype == 1) v = static_cast<float>(reinterpret_cast<const long long*>(src)[t]);
  else if (dtype == 2) v = reinterpret_cast<const float*>(src)[t];
  else if (dtype == 3) v = static_cast<float>(reinterpret_cast<const int*>(src)[t]);
  else if (dtype == 4) v = static_cast<float>(reinterpret_cast<const unsigned char*>(src)[t]);
  dst[t] = v != 0.f;
  if (dstf) dstf[t] = v;
}

// x = table[ids]*sqrt(D) (pre-scaled at load) + pe[l]   (models/text_encoder.py:504-512)
__global__ void embed_kernel(const long long* __restrict__ ids, const float4* __restrict__ table,
                             const float4* __restrict__ pe, float4* __restrict__ dst, int T, int L, int D4, int V) {
  pdl_launch_dependents();
  pdl_wait();
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T * D4) return;
  const int tok = t / D4, d = t - tok * D4;
  long long id = ids[tok];
  id = id < 0 ? 0 : (id >= V ? V - 1 : id);
  const float4 e = table[static_cast<size_t>(id) * D4 + d];
  const float4 p = pe[static_cast<size_t>(tok % L) * D4 + d];
  dst[t] = make_float4(e.x + p.x, e.y + p.y, e.z + p.z, e.w + p.w);
}

// LayerNorm over D = 256, one warp per row (biased variance, eps inside the sqrt).  mode 1 is the
// image projector's variant: source rows are the valid pixels of the 7x7 (+pad) grid and the
// learned position embedding is added after the affine (models/fusion.py:98-112).
// One LayerNorm-256 row held by a warp (8 values per lane: columns 4*lane.. and 128 + 4*lane..): statistics, affine.
__device__ __forceinline__ void ln256_apply(const float (&x)[8], const float4& g0, const float4& g1, const float4& b0,
                                            const float4& b1, float eps, float (&y)[8]) {
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < 8; ++k) s += x[k];
  const float mean = warp_sum(s) * (1.f / 256.f);
  float v[8], q = 0.f;
#pragma unroll
  for (int k = 0; k < 8; ++k) { v[k] = x[k] - mean; q += v[k] * v[k]; }
  const float rstd = rsqrtf(warp_sum(q) * (1.f / 256.f) + eps);
  const float g[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
  const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
  for (int k = 0; k < 8; ++k) y[k] = v[k] * rstd * g[k] + bb[k];
}
// Store a row: rnd 0 = fp32, 1 = tf32-rounded fp32, 2 = fp16 (operand of an fp16 Linear).
__device__ __forceinline__ void ln256_store(float* dst, int row, int lane, int rnd, float (&y)[8]) {
  if (rnd == 2) {   // 8 bytes per float4
    uint2* o2 = reinterpret_cast<uint2*>(reinterpret_cast<__half*>(dst) + static_cast<size_t>(row) * 256);
    o2[lane] = make_uint2(pack_f16x2(y[0], y[1]), pack_f16x2(y[2], y[3]));
    o2[32 + lane] = make_uint2(pack_f16x2(y[4], y[5]), pack_f16x2(y[6], y[7]));
    return;
  }
  float4* o4 = reinterpret_cast<float4*>(dst + static_cast<size_t>(row) * 256);
  if (rnd) {
    o4[lane] = make_float4(round_tf32_rna(y[0]), round_tf32_rna(y[1]), round_tf32_rna(y[2]), round_tf32_rna(y[3]));
    o4[32 + lane] = make_float4(round_tf32_rna(y[4]), round_tf32_rna(y[5]), round_tf32_rna(y[6]), round_tf32_rna(y[7]));
  } else {
    o4[lane] = make_float4(y[0], y[1], y[2], y[3]);
    o4[32 + lane] = make_float4(y[4], y[5], y[6], y[7]);
  }
}

// Up to two further LayerNorms of the (unrounded) first output in the same launch: the final text norm + the first
// cross-attention layer's query norm (text_encoder.py:522, cross_attention.py:265), the projector norm + the key/value
// norms of the cross-attention layers (fusion.py:98-112, cross_attention.py:266).
struct LnExtra {
  const float *gamma2, *beta2, *gamma3, *beta3;
  float *dst2, *dst3;
  int rnd2, rnd3;
};

__global__ void layernorm256_kernel(const float* __restrict__ src, const float* __restrict__ gamma,
                                    const float* __restrict__ beta, float* __restrict__ dst,
                                    const float* __restrict__ pos, int rows, int ld, int mode, int rnd, int S, int Pg,
                                    int RPIg, float eps, const LnExtra ex) {
  pdl_launch_dependents();
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  // gamma / beta are weights: fetch them before waiting for the kernel that produces the rows
  const float4 g0 = __ldg(reinterpret_cast<const float4*>(gamma) + lane), g1 = __ldg(reinterpret_cast<const float4*>(gamma) + 32 + lane);
  const float4 b0 = __ldg(reinterpret_cast<const float4*>(beta) + lane), b1 = __ldg(reinterpret_cast<const float4*>(beta) + 32 + lane);
  pdl_wait();
  if (row >= rows) return;
  size_t srow = row;
  int pix = 0;
  if (mode == 1) {
    const int n = row / (S * S);
    pix = row - n * S * S;
    srow = static_cast<size_t>(n) * RPIg + (pix / S) * Pg + (pix % S);
  }
  const float4* x4 = reinterpret_cast<const float4*>(src + srow * ld);
  const float4 a = x4[lane], b = x4[32 + lane];
  const float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
  float y[8];
  ln256_apply(v, g0, g1, b0, b1, eps, y);
  if (mode == 1 && pos) {
    const float4 p0 = reinterpret_cast<const float4*>(pos + static_cast<size_t>(pix) * 256)[lane];
    const float4 p1 = reinterpret_cast<const float4*>(pos + static_cast<size_t>(pix) * 256)[32 + lane];
    y[0] += p0.x; y[1] += p0.y; y[2] += p0.z; y[3] += p0.w;
    y[4] += p1.x; y[5] += p1.y; y[6] += p1.z; y[7] += p1.w;
  }
  if (ex.gamma2 != nullptr) {
    float z[8];
    ln256_apply(y, __ldg(reinterpret_cast<const float4*>(ex.gamma2) + lane), __ldg(reinterpret_cast<const float4*>(ex.gamma2) + 32 + lane),
                __ldg(reinterpret_cast<const float4*>(ex.beta2) + lane), __ldg(reinterpret_cast<const float4*>(ex.beta2) + 32 + lane), eps, z);
    ln256_store(ex.dst2, row, lane, ex.rnd2, z);
  }
  if (ex.gamma3 != nullptr) {
    float z[8];
    ln256_apply(y, __ldg(reinterpret_cast<const float4*>(ex.gamma3) + lane), __ldg(reinterpret_cast<const float4*>(ex.gamma3) + 32 + lane),
                __ldg(reinterpret_cast<const float4*>(ex.beta3) + lane), __ldg(reinterpret_cast<const float4*>(ex.beta3) + 32 + lane), eps, z);
    ln256_store(ex.dst3, row, lane, ex.rnd3, z);
  }
  ln256_store(dst, row, lane, rnd, y);
}

// EMBED with the first encoder layer's LayerNorm and the mask normalisation in the same launch (warp per token):
// x = table[id] + pe[position] -> dst (the fp32 residual stream); LN(x) -> ln_dst; the token's mask element -> int32 key mask
// + float pooling weight (text_encoder.py:504-512, :373; fusion.py:299-312).
__global__ void embed_ln_kernel(const long long* __restrict__ ids, const float* __restrict__ table, const float* __restrict__ pe,
                                float* __restrict__ dst, const float* __restrict__ gamma, const float* __restrict__ beta,
                                float* __restrict__ ln_dst, int T, int L, int V, int rnd, float eps,
                                const void* __restrict__ mask_src, int* __restrict__ mask_dst, float* __restrict__ mask_dstf,
                                int mask_dtype) {
  pdl_launch_dependents();
  const int tok = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  const float4 g0 = __ldg(reinterpret_cast<const float4*>(gamma) + lane), g1 = __ldg(reinterpret_cast<const float4*>(gamma) + 32 + lane);
  const float4 b0 = __ldg(reinterpret_cast<const float4*>(beta) + lane), b1 = __ldg(reinterpret_cast<const float4*>(beta) + 32 + lane);
  pdl_wait();
  if (tok >= T) return;
  if (lane == 0 && mask_dst != nullptr) {
    float m = 1.f;
    if (mask_dtype == 1) m = static_cast<float>(reinterpret_cast<const long long*>(mask_src)[tok]);
    else if (mask_dtype == 2) m = reinterpret_cast<const float*>(mask_src)[tok];
    else if (mask_dtype == 3) m = static_cast<float>(reinterpret_cast<const int*>(mask_src)[tok]);
    else if (mask_dtype == 4) m = static_cast<float>(reinterpret_cast<const unsigned char*>(mask_src)[tok]);
    mask_dst[tok] = m != 0.f;
    if (mask_dstf) mask_dstf[tok] = m;
  }
  long long id = ids[tok];
  id = id < 0 ? 0 : (id >= V ? V - 1 : id);
  const float4* e4 = reinterpret_cast<const float4*>(table + static_cast<size_t>(id) * 256);
  const float4* p4 = reinterpret_cast<const float4*>(pe + static_cast<size_t>(tok % L) * 256);
  const float4 e0 = __ldg(e4 + lane), e1 = __ldg(e4 + 32 + lane), p0 = __ldg(p4 + lane), p1 = __ldg(p4 + 32 + lane);
  const float x[8] = {e0.x + p0.x, e0.y + p0.y, e0.z + p0.z, e0.w + p0.w, e1.x + p1.x, e1.y + p1.y, e1.z + p1.z, e1.w + p1.w};
  float4* o4 = reinterpret_cast<float4*>(dst + static_cast<size_t>(tok) * 256);
  o4[lane] = make_float4(x[0], x[1], x[2], x[3]);
  o4[32 + lane] = make_float4(x[4], x[5], x[6], x[7]);
  float y[8];
  ln256_apply(x, g0, g1, b0, b1, eps, y);
  ln256_store(ln_dst, tok, lane, rnd, y);
}

constexpr int kHd = 32;
constexpr int kAttnWarps = 4;

// ------------------------------------------------------------------------------------------------
// Attention core, one WARP per (pair, head): softmax(Q K^T / sqrt(32) [+ key mask]) V with head_dim 32, up
// to 64 queries (blocks of 32) and up to 64 keys.  Self-attention (models/text_encoder.py:229-259; keys
// with mask == 0 get -inf, a fully masked row yields NaN exactly like the reference, SURVEY T5) and
// cross-attention over the 49 image tokens (models/cross_attention.py:164-197, no mask) share it.
// S = Q K^T and O = P V run on mma.sync m16n8k8 with the 3xTF32 split (x = hi + lo; lo*hi + hi*lo + hi*hi:
// fp32-level accuracy, the parity budget has no room for a plain tf32 attention); softmax stays in fp32
// registers on the accumulator fragments.  CUDA-core versions measured 2-4x slower (lane per key: shuffle
// bound, 57 us for the cross attention of 256 pairs; lane per query: LDS.128 broadcast bound, 69 us; this
// kernel 31 us).  NT = key tiles of 8.
// x = hi + lo with both parts exact tf32 values: hi keeps the top 19 bits (truncation), x - hi is exact in fp32 and
// is truncated again (loses < 2^-21 |x|).  Three ALU instructions; cvt.rna.tf32.f32 is emulated on sm_100a (~5
// instructions each) and made the splits half of this kernel's instruction count (ncu source view).
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(x) & 0xFFFFE000u;
  lo = __float_as_uint(x - __uint_as_float(hi)) & 0xFFFFE000u;
}
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void mma_3xtf32(float (&d)[4], const uint32_t (&ah)[4], const uint32_t (&al)[4], uint32_t bh0,
                                           uint32_t bh1, uint32_t bl0, uint32_t bl1) {
  mma_tf32(d, al, bh0, bh1);
  mma_tf32(d, ah, bl0, bl1);
  mma_tf32(d, ah, bh0, bh1);
}

constexpr int kKs = 36, kVs = 40;                       // padded row strides (floats): conflict-free fragment loads
__host__ __device__ constexpr int attn_mma_kreg(int nt) {           // K rows, later the probability tile [32][nt*8+4]
  return nt * 8 * kKs > 32 * (nt * 8 + 4) ? nt * 8 * kKs : 32 * (nt * 8 + 4);
}
__host__ __device__ constexpr int attn_mma_warp_floats(int nt) { return attn_mma_kreg(nt) + nt * 8 * kVs; }

template <int NT>
__global__ void __launch_bounds__(kAttnWarps * 32)
attn_mma_kernel(const float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v,
                const int* __restrict__ mask, float* __restrict__ out, float* __restrict__ weights, int n_units,
                int H, int L, int T, int ld_q, int ld_kv, int no_round, int q_per_kv) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ __align__(16) float sm[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int unit = blockIdx.x * kAttnWarps + warp;     // (pair, head)
  if (unit >= n_units) return;
  const int b = unit / H, h = unit - b * H;
  constexpr int PS = NT * 8 + 4;                        // probability tile row stride
  float* Ks = sm + warp * attn_mma_warp_floats(NT);
  float* Ps = Ks;
  float* Vs = Ks + attn_mma_kreg(NT);
  const float* qb = q + static_cast<size_t>(b) * L * ld_q + h * kHd;
  const int bkv = b / q_per_kv;                         // q_per_kv consecutive queries share one image's K / V
  const float* kb = k + static_cast<size_t>(bkv) * T * ld_kv + h * kHd;
  const float* vb = v + static_cast<size_t>(bkv) * T * ld_kv + h * kHd;
  // K / V rows go global -> shared with cp.async (all 16-byte pieces of the head in flight at once; rows beyond T
  // are zero-filled through the src-size operand).  A register-staged loop serialised 14 + 14 DRAM/L2 round trips
  // per warp and was 1/3 of the kernel's stall samples (ncu source view, profiles/r01_h_*).
  auto stage_rows = [&](float* dst, int stride, const float* src) {
    for (int i = lane; i < NT * 8 * 8; i += 32) {
      const int r = i >> 3, c4 = i & 7;
      const float* g = src + static_cast<size_t>(r < T ? r : 0) * ld_kv + c4 * 4;
      const uint32_t d = static_cast<uint32_t>(__cvta_generic_to_shared(dst + r * stride + c4 * 4));
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(g), "r"(r < T ? 16 : 0) : "memory");
    }
  };
  stage_rows(Vs, kVs, vb);
  float mb[NT][2];                                      // additive key mask of this lane's score columns
#pragma unroll
  for (int n = 0; n < NT; ++n)
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int j = n * 8 + 2 * t + e;
      mb[n][e] = (j < T && (mask == nullptr || mask[b * T + j] != 0)) ? 0.f : -INFINITY;   // self-attention only (q_per_kv = 1)
    }
  const float scale = rsqrtf(static_cast<float>(kHd));
  for (int l0 = 0; l0 < L; l0 += 32) {
    __syncwarp();
    stage_rows(Ks, kKs, kb);                            // K rows (the region is reused for P below)
    asm volatile("cp.async.commit_group;" ::: "memory");
    // Q fragments (rows g, g+8 of each 16-row tile; dims t, t+4 of each 8-wide k step), pre-split
    uint32_t qh[2][4][4], ql[2][4][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int ks = 0; ks < 4; ++ks)
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int row = l0 + mt * 16 + g + (e & 1) * 8, col = ks * 8 + t + (e >> 1) * 4;
          const float x = row < L ? __ldg(qb + static_cast<size_t>(row) * ld_q + col) : 0.f;
          split_tf32(x, qh[mt][ks][e], ql[mt][ks][e]);
        }
    asm volatile("cp.async.wait_group 0;" ::: "memory");   // this lane's K (and, first pass, V) pieces have landed
    __syncwarp();
    float sacc[2][NT][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int n = 0; n < NT; ++n)
#pragma unroll
        for (int e = 0; e < 4; ++e) sacc[mt][n][e] = 0.f;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks)
#pragma unroll
      for (int n = 0; n < NT; ++n) {
        uint32_t bh0, bl0, bh1, bl1;
        split_tf32(Ks[(n * 8 + g) * kKs + ks * 8 + t], bh0, bl0);
        split_tf32(Ks[(n * 8 + g) * kKs + ks * 8 + t + 4], bh1, bl1);
        mma_3xtf32(sacc[0][n], qh[0][ks], ql[0][ks], bh0, bh1, bl0, bl1);
        mma_3xtf32(sacc[1][n], qh[1][ks], ql[1][ks], bh0, bh1, bl0, bl1);
      }
    __syncwarp();                                       // every lane is done with K: the region becomes P
    // softmax on the fragments: accumulator e -> row (e >> 1) * 8 + g of the tile, column 2t + (e & 1)
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int hf = 0; hf < 2; ++hf) {
        float mx = -INFINITY;
#pragma unroll
        for (int n = 0; n < NT; ++n)
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const float sv = sacc[mt][n][hf * 2 + e] * scale + mb[n][e];
            sacc[mt][n][hf * 2 + e] = sv;
            mx = fmaxf(mx, sv);
          }
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
        float sum = 0.f;                                // exp(-inf - -inf) = NaN reproduces a fully masked row
#pragma unroll
        for (int n = 0; n < NT; ++n)
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const float pv = expf(sacc[mt][n][hf * 2 + e] - mx);
            sacc[mt][n][hf * 2 + e] = pv;
            sum += pv;
          }
        sum += __shfl_xor_sync(0xffffffffu, sum, 1);
        sum += __shfl_xor_sync(0xffffffffu, sum, 2);
        const float inv = 1.f / sum;
        float* prow = Ps + (mt * 16 + hf * 8 + g) * PS + 2 * t;
#pragma unroll
        for (int n = 0; n < NT; ++n)
          *reinterpret_cast<float2*>(prow + n * 8) = make_float2(sacc[mt][n][hf * 2] * inv, sacc[mt][n][hf * 2 + 1] * inv);
      }
    __syncwarp();
    if (weights) {
      const int rows = min(32, L - l0);
      float* wb = weights + ((static_cast<size_t>(b) * H + h) * L + l0) * T;
      for (int i = lane; i < rows * T; i += 32) wb[i] = Ps[(i / T) * PS + (i % T)];
    }
    float oacc[2][4][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int n = 0; n < 4; ++n)
#pragma unroll
        for (int e = 0; e < 4; ++e) oacc[mt][n][e] = 0.f;
#pragma unroll
    for (int kk = 0; kk < NT; ++kk) {
      uint32_t ah[2][4], al[2][4];
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int e = 0; e < 4; ++e)
          split_tf32(Ps[(mt * 16 + g + (e & 1) * 8) * PS + kk * 8 + t + (e >> 1) * 4], ah[mt][e], al[mt][e]);
#pragma unroll
      for (int n = 0; n < 4; ++n) {
        uint32_t bh0, bl0, bh1, bl1;
        split_tf32(Vs[(kk * 8 + t) * kVs + n * 8 + g], bh0, bl0);
        split_tf32(Vs[(kk * 8 + t + 4) * kVs + n * 8 + g], bh1, bl1);
        mma_3xtf32(oacc[0][n], ah[0], al[0], bh0, bh1, bl0, bl1);
        mma_3xtf32(oacc[1][n], ah[1], al[1], bh0, bh1, bl0, bl1);
      }
    }
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int hf = 0; hf < 2; ++hf) {
        const int row = l0 + mt * 16 + hf * 8 + g;
        if (row < L) {
          float* orow = out + (static_cast<size_t>(b) * L + row) * (H * kHd) + h * kHd + 2 * t;
#pragma unroll
          for (int n = 0; n < 4; ++n) {                 // operand of W_o: fp16 (2), unrounded for the 3xTF32 split (1), tf32 (0)
            const float o0 = oacc[mt][n][hf * 2], o1 = oacc[mt][n][hf * 2 + 1];
            if (no_round == 2) {
              __half* hrow = reinterpret_cast<__half*>(out) + (static_cast<size_t>(b) * L + row) * (H * kHd) + h * kHd + 2 * t;
              *reinterpret_cast<uint32_t*>(hrow + n * 8) = pack_f16x2(o0, o1);
            } else {
              *reinterpret_cast<float2*>(orow + n * 8) = no_round ? make_float2(o0, o1)
                                                                  : make_float2(round_tf32_rna(o0), round_tf32_rna(o1));
            }
          }
        }
      }
  }
}

typedef void (*AttnFn)(const float*, const float*, const float*, const int*, float*, float*, int, int, int, int, int, int, int,
                       int);

static int launch_attn(const float* q, const float* k, const float* v, const int* mask, float* out, float* weights, int B,
                       int H, int L, int T, int ld_q, int ld_kv, int no_round, int q_per_kv, cudaStream_t st) {
  VQA_REQUIRE(q_per_kv >= 1 && B % q_per_kv == 0, VQA_E_INVALID, "attention: the batch must be a multiple of q_per_kv");
  const int nt = (T + 7) / 8;
  VQA_REQUIRE(nt >= 1 && nt <= 8, VQA_E_INVALID, "attention: 1..64 keys");
  const int ntt = nt <= 3 ? 3 : nt <= 4 ? 4 : nt <= 7 ? 7 : 8;
  AttnFn fn = ntt == 3 ? static_cast<AttnFn>(&attn_mma_kernel<3>) : ntt == 4 ? static_cast<AttnFn>(&attn_mma_kernel<4>)
            : ntt == 7 ? static_cast<AttnFn>(&attn_mma_kernel<7>) : static_cast<AttnFn>(&attn_mma_kernel<8>);
  const size_t smem = static_cast<size_t>(kAttnWarps) * attn_mma_warp_floats(ntt) * sizeof(float);
  // cudaFuncSetAttribute is per device (context): remember it per (device, instantiation)
  static bool attr_set[kMaxDevices][9] = {};
  int dev = 0;
  VQA_CUDA_OK(cudaGetDevice(&dev));
  if (dev < 0 || dev >= kMaxDevices || !attr_set[dev][ntt]) {
    VQA_CUDA_OK(cudaFuncSetAttribute(reinterpret_cast<const void*>(fn), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     static_cast<int>(smem)));
    if (dev >= 0 && dev < kMaxDevices) attr_set[dev][ntt] = true;
  }
  VQA_CUDA_OK(vqa_launch(fn, dim3((B * H + kAttnWarps - 1) / kAttnWarps), dim3(kAttnWarps * 32), smem, st, q, k, v, mask, out,
                         weights, B * H, H, L, T, ld_q, ld_kv, no_round, q_per_kv));
  VQA_LAUNCH_OK("attn_mma_kernel");
  return VQA_OK;
}

// ------------------------------------------------------------------------------------------------
// Fusion tail, one pair per CTA, D = 256 = blockDim (models/fusion.py:299-326, :159-166):
//   phase 1: masked mean pools of the cross-attended and text features (denominator clamp(min=1)),
//            written as att_pooled / txt_pooled and as the tf32 row [att;txt] of the gate GEMM
//   phase 2: g = sigmoid(pre) with pre = W[att;txt]+b from that GEMM, g*att+(1-g)*txt, output LayerNorm
//   phase 0: no gating: att+txt, output LayerNorm (pools computed in place)
__global__ void __launch_bounds__(256)
pool_gate_ln_kernel(const float* __restrict__ xatt, const float* __restrict__ text, const float* __restrict__ mask,
                    const float* __restrict__ pre, const float* __restrict__ gamma, const float* __restrict__ beta,
                    float* __restrict__ fused, float* __restrict__ att_pooled, float* __restrict__ txt_pooled,
                    float* __restrict__ cat, int L, int phase, int no_round, float eps) {
  pdl_launch_dependents();
  const float gam = __ldg(gamma + threadIdx.x), bet = __ldg(beta + threadIdx.x);   // weights: before the dependency wait
  pdl_wait();
  constexpr int D = 256;
  __shared__ float red[16];
  const int b = blockIdx.x, d = threadIdx.x;
  const int warp = d >> 5, lane = d & 31;
  float ap, tp;
  if (phase != 2) {
    float cnt = 0.f, sa = 0.f, st = 0.f;
#pragma unroll 4
    for (int l = 0; l < L; ++l) {
      const float m = mask ? mask[b * L + l] : 1.f;   // attention_mask.float() as pooling weight
      cnt += m;
      sa += xatt[(static_cast<size_t>(b) * L + l) * D + d] * m;
      st += text[(static_cast<size_t>(b) * L + l) * D + d] * m;
    }
    const float den = fmaxf(cnt, 1.f);
    ap = sa / den;
    tp = st / den;
    att_pooled[static_cast<size_t>(b) * D + d] = ap;
    txt_pooled[static_cast<size_t>(b) * D + d] = tp;
    if (phase == 1) {
      if (no_round == 2) {   // fp16 operand of the gate GEMM
        __half* hc = reinterpret_cast<__half*>(cat) + static_cast<size_t>(b) * 2 * D;
        hc[d] = __float2half_rn(ap);
        hc[D + d] = __float2half_rn(tp);
      } else {
        cat[static_cast<size_t>(b) * 2 * D + d] = no_round ? ap : round_tf32_rna(ap);
        cat[static_cast<size_t>(b) * 2 * D + D + d] = no_round ? tp : round_tf32_rna(tp);
      }
      return;
    }
  } else {
    ap = att_pooled[static_cast<size_t>(b) * D + d];
    tp = txt_pooled[static_cast<size_t>(b) * D + d];
  }
  float f;
  if (phase == 2) {
    const float g = 1.f / (1.f + expf(-pre[static_cast<size_t>(b) * D + d]));
    f = g * ap + (1.f - g) * tp;
  } else {
    f = ap + tp;
  }
  // block LayerNorm over 256 values (8 warps)
  const float s = warp_sum(f);
  if (lane == 0) red[warp] = s;
  __syncthreads();
  float mean = 0.f;
  for (int w = 0; w < 8; ++w) mean += red[w];
  const float c = f - mean * (1.f / D);
  const float q = warp_sum(c * c);
  if (lane == 0) red[8 + warp] = q;
  __syncthreads();
  float var = 0.f;
  for (int w = 0; w < 8; ++w) var += red[8 + w];
  var *= (1.f / D);
  const float y = c * rsqrtf(var + eps) * gam + bet;
  fused[static_cast<size_t>(b) * D + d] = y;
  if (no_round == 2 && cat != nullptr)   // phases 0 / 2: fp16 copy of the fused feature = operand of the first head Linear
    reinterpret_cast<__half*>(cat)[static_cast<size_t>(b) * D + d] = __float2half_rn(y);
}

// softmax over N answers + top-k (k <= 128) in rank_before's order, torch.topk's with ties broken towards the lower index
// (models/vqa_model.py:336-337, api/inference.py:231-234).
__global__ void softmax_topk_kernel(const float* __restrict__ logits, long long* __restrict__ idx,
                                    float* __restrict__ probs, int N, int k, int ld) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ float sm[];  // vals[N], red[64], taken bits[(N + 31) / 32]
  float* vals = sm;
  float* red = sm + N;
  int* redi = reinterpret_cast<int*>(red + 32);
  uint32_t* flags = reinterpret_cast<uint32_t*>(red + 64);
  auto taken = [&](int i) { return (flags[i >> 5] >> (i & 31)) & 1u; };
  const int b = blockIdx.x, tid = threadIdx.x, nw = blockDim.x >> 5;
  const float* row = logits + static_cast<size_t>(b) * ld;
  float m = -INFINITY;
  for (int i = tid; i < (N + 31) / 32; i += blockDim.x) flags[i] = 0u;
  for (int i = tid; i < N; i += blockDim.x) { vals[i] = row[i]; m = fmaxf(m, vals[i]); }
  m = warp_max(m);
  if ((tid & 31) == 0) red[tid >> 5] = m;
  __syncthreads();
  m = -INFINITY;
  for (int w = 0; w < nw; ++w) m = fmaxf(m, red[w]);
  __syncthreads();
  float s = 0.f;
  for (int i = tid; i < N; i += blockDim.x) s += expf(vals[i] - m);
  s = warp_sum(s);
  if ((tid & 31) == 0) red[tid >> 5] = s;
  __syncthreads();
  s = 0.f;
  for (int w = 0; w < nw; ++w) s += red[w];
  __syncthreads();
  // Selection order: NaN ranks above everything (torch.topk's order), so a row of NaNs -- the reference's result for a
  // fully masked question, models/text_encoder.py:244 -- yields indices 0..k-1 with NaN probabilities instead of no winner
  // at all; a picked entry is retired through the `taken` flag, never by its value.
  for (int t = 0; t < k; ++t) {
    float best = -INFINITY;
    int bi = 0x7fffffff;
    for (int i = tid; i < N; i += blockDim.x) {
      const float v = vals[i];
      if (!taken(i) && rank_before(v, i, best, bi)) { best = v; bi = i; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ob = __shfl_xor_sync(0xffffffffu, best, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (rank_before(ob, oi, best, bi)) { best = ob; bi = oi; }
    }
    if ((tid & 31) == 0) { red[tid >> 5] = best; redi[tid >> 5] = bi; }
    __syncthreads();
    if (tid == 0) {
      float bb = red[0];
      int ii = redi[0];
      for (int w = 1; w < nw; ++w)
        if (rank_before(red[w], redi[w], bb, ii)) { bb = red[w]; ii = redi[w]; }
      if (ii < 0 || ii >= N) ii = t < N ? t : N - 1;      // cannot happen with k <= N; never index out of the row
      idx[static_cast<size_t>(b) * k + t] = ii;
      probs[static_cast<size_t>(b) * k + t] = expf(vals[ii] - m) / s;
      flags[ii >> 5] |= 1u << (ii & 31);
    }
    __syncthreads();
  }
}

inline unsigned blocks_for(long long n, int threads) { return static_cast<unsigned>((n + threads - 1) / threads); }

}  // namespace

// ================================================================================================
// launchers
#define PTR(T, k) reinterpret_cast<T>(vqa_resolve(op.p[k], ext, n_ext))

int run_misc_op(const VqaOp& op, const uint64_t* ext, int n_ext, cudaStream_t st) {
  const int32_t* I = op.i;
  switch (op.kind) {
    case VQA_OP_INGEST: {
      const int rows = I[INGEST_I_rows];
      VQA_REQUIRE(I[INGEST_I_HW] == 224 && I[INGEST_I_P] == 114, VQA_E_INVALID, "ingest: only 224x224 inputs");
      const void* src = PTR(const void*, INGEST_P_src);
      VQA_REQUIRE(src != nullptr, VQA_E_INVALID, "ingest: null images");
      VQA_REQUIRE((reinterpret_cast<uintptr_t>(src) & 7) == 0 || I[INGEST_I_mode] == 1, VQA_E_ALIGN,
                  "ingest: fp32 images must be 8-byte aligned");
      VQA_REQUIRE((reinterpret_cast<uintptr_t>(src) & 1) == 0, VQA_E_ALIGN, "ingest: uint8 images must be 2-byte aligned");
      VQA_CUDA_OK(vqa_launch(ingest_kernel, dim3(blocks_for(rows, 256)), dim3(256), 0, st, src, PTR(uint4*, INGEST_P_dst), I[INGEST_I_B],
                                                            I[INGEST_I_mode], I[INGEST_I_P], rows, I[INGEST_I_ones], I[INGEST_I_f32]));
      VQA_LAUNCH_OK("ingest_kernel");
      return VQA_OK;
    }
    case VQA_OP_MAXPOOL: {
      if (I[MAXPOOL_I_f32]) {
        const int C4 = I[MAXPOOL_I_C] / 4;
        const long long tot = static_cast<long long>(I[MAXPOOL_I_B]) * I[MAXPOOL_I_RPIout] * C4;
        VQA_CUDA_OK(vqa_launch(maxpool_f32_kernel, dim3(blocks_for(tot, 256)), dim3(256), 0, st,
            PTR(const float4*, MAXPOOL_P_src), PTR(float4*, MAXPOOL_P_dst), I[MAXPOOL_I_B], C4, I[MAXPOOL_I_Hin],
            I[MAXPOOL_I_Win], I[MAXPOOL_I_Pin], I[MAXPOOL_I_RPIin], I[MAXPOOL_I_Hout], I[MAXPOOL_I_Wout],
            I[MAXPOOL_I_Pout], I[MAXPOOL_I_RPIout]));
        VQA_LAUNCH_OK("maxpool_f32_kernel");
        return VQA_OK;
      }
      const int C8 = I[MAXPOOL_I_C] / 8;
      const long long total = static_cast<long long>(I[MAXPOOL_I_B]) * I[MAXPOOL_I_RPIout] * C8;
      VQA_CUDA_OK(vqa_launch(maxpool_kernel, dim3(blocks_for(total, 256)), dim3(256), 0, st, 
          PTR(const uint4*, MAXPOOL_P_src), PTR(uint4*, MAXPOOL_P_dst), I[MAXPOOL_I_B], C8, I[MAXPOOL_I_Hin],
          I[MAXPOOL_I_Win], I[MAXPOOL_I_Pin], I[MAXPOOL_I_RPIin], I[MAXPOOL_I_Hout], I[MAXPOOL_I_Wout],
          I[MAXPOOL_I_Pout], I[MAXPOOL_I_RPIout]));
      VQA_LAUNCH_OK("maxpool_kernel");
      return VQA_OK;
    }
    case VQA_OP_SE_SQUEEZE: {
      const int C8 = I[SE_SQUEEZE_I_C] / 8;
      VQA_REQUIRE(C8 >= 1 && C8 <= 256, VQA_E_INVALID, "se_squeeze: C out of range");
      const int threads = 256 >= C8 ? 256 / C8 * C8 : C8;
      const size_t smem = static_cast<size_t>(threads) * 8 * sizeof(float);
      const int slices = I[SE_SQUEEZE_I_S];
      VQA_REQUIRE(slices >= 1 && slices <= 64, VQA_E_INVALID, "se_squeeze: bad slice count");
      VQA_CUDA_OK(vqa_launch(se_squeeze_kernel, dim3(dim3(I[SE_SQUEEZE_I_B], slices)), dim3(threads), smem, st, PTR(const uint4*, SE_SQUEEZE_P_src),
                                                                  PTR(float*, SE_SQUEEZE_P_sums), C8, I[SE_SQUEEZE_I_H],
                                                                  I[SE_SQUEEZE_I_W], I[SE_SQUEEZE_I_P],
                                                                  I[SE_SQUEEZE_I_RPI]));
      VQA_LAUNCH_OK("se_squeeze_kernel");
      return VQA_OK;
    }
    case VQA_OP_SE_EXCITE: {
      const int C = I[SE_EXCITE_I_C], R = I[SE_EXCITE_I_R];
      VQA_CUDA_OK(vqa_launch(se_excite_kernel, dim3(I[SE_EXCITE_I_B]), dim3(256), (C + R) * sizeof(float), st, 
          PTR(const float*, SE_EXCITE_P_sums), PTR(const float*, SE_EXCITE_P_w1), PTR(const float*, SE_EXCITE_P_w2),
          PTR(float*, SE_EXCITE_P_scale), C, R, I[SE_EXCITE_I_S], 1.f / static_cast<float>(I[SE_EXCITE_I_HW])));
      VQA_LAUNCH_OK("se_excite_kernel");
      return VQA_OK;
    }
    case VQA_OP_SPATIAL_MAP: {
      const int C = I[SPATIAL_MAP_I_C], HW = I[SPATIAL_MAP_I_H] * I[SPATIAL_MAP_I_W];
      const size_t smem = (2 * HW + C) * sizeof(float);
      VQA_REQUIRE(smem <= 48 * 1024, VQA_E_INVALID, "spatial_map: feature map too large");
      VQA_CUDA_OK(vqa_launch(spatial_map_kernel, dim3(I[SPATIAL_MAP_I_B]), dim3(256), smem, st, 
          PTR(const uint4*, SPATIAL_MAP_P_src), PTR(const float*, SPATIAL_MAP_P_scale),
          PTR(const float*, SPATIAL_MAP_P_wconv), PTR(float*, SPATIAL_MAP_P_att), C / 8, I[SPATIAL_MAP_I_H],
          I[SPATIAL_MAP_I_W], I[SPATIAL_MAP_I_P], I[SPATIAL_MAP_I_RPI], I[SPATIAL_MAP_I_ksize]));
      VQA_LAUNCH_OK("spatial_map_kernel");
      return VQA_OK;
    }
    case VQA_OP_SCALE_RELAYOUT: {
      const int C8 = I[SCALE_RELAYOUT_I_C] / 8, mode = I[SCALE_RELAYOUT_I_mode];
      const long long rows = mode ? 4LL * I[SCALE_RELAYOUT_I_phase_rows]
                                  : static_cast<long long>(I[SCALE_RELAYOUT_I_B]) * I[SCALE_RELAYOUT_I_RPIo];
      VQA_CUDA_OK(vqa_launch(scale_relayout_kernel, dim3(blocks_for(rows * C8, 256)), dim3(256), 0, st, 
          PTR(const uint4*, SCALE_RELAYOUT_P_src), PTR(const float*, SCALE_RELAYOUT_P_scale),
          PTR(const float*, SCALE_RELAYOUT_P_att), PTR(uint4*, SCALE_RELAYOUT_P_dst), I[SCALE_RELAYOUT_I_B], C8,
          I[SCALE_RELAYOUT_I_H], I[SCALE_RELAYOUT_I_W], I[SCALE_RELAYOUT_I_P], I[SCALE_RELAYOUT_I_RPI], mode,
          I[SCALE_RELAYOUT_I_Po], I[SCALE_RELAYOUT_I_RPIo], I[SCALE_RELAYOUT_I_phase_rows]));
      VQA_LAUNCH_OK("scale_relayout_kernel");
      return VQA_OK;
    }
    case VQA_OP_GRID_TO_NCHW: {
      const long long total = static_cast<long long>(I[GRID_TO_NCHW_I_B]) * I[GRID_TO_NCHW_I_C] * I[GRID_TO_NCHW_I_H] *
                              I[GRID_TO_NCHW_I_W];
      VQA_CUDA_OK(vqa_launch(grid_to_nchw_kernel, dim3(blocks_for(total, 256)), dim3(256), 0, st, 
          PTR(const void*, GRID_TO_NCHW_P_src), PTR(float*, GRID_TO_NCHW_P_dst), I[GRID_TO_NCHW_I_B],
          I[GRID_TO_NCHW_I_C], I[GRID_TO_NCHW_I_H], I[GRID_TO_NCHW_I_W], I[GRID_TO_NCHW_I_P], I[GRID_TO_NCHW_I_RPI],
          I[GRID_TO_NCHW_I_f32]));
      VQA_LAUNCH_OK("grid_to_nchw_kernel");
      return VQA_OK;
    }
    case VQA_OP_STAGE_TAIL: {
      StageTailParams q;
      q.src = PTR(const uint4*, STAGE_TAIL_P_src);
      q.w1 = PTR(const float*, STAGE_TAIL_P_w1);
      q.w2 = PTR(const float*, STAGE_TAIL_P_w2);
      q.wconv = PTR(const float*, STAGE_TAIL_P_wconv);
      q.dst = PTR(uint4*, STAGE_TAIL_P_dst);
      q.scale_out = PTR(float*, STAGE_TAIL_P_scale);
      q.att_out = PTR(float*, STAGE_TAIL_P_att);
      const int C = I[STAGE_TAIL_I_C];
      q.C8 = C / 8; q.H = I[STAGE_TAIL_I_H]; q.W = I[STAGE_TAIL_I_W]; q.P = I[STAGE_TAIL_I_P]; q.RPI = I[STAGE_TAIL_I_RPI];
      q.R = I[STAGE_TAIL_I_R]; q.ks = I[STAGE_TAIL_I_ks]; q.mode = I[STAGE_TAIL_I_mode]; q.Po = I[STAGE_TAIL_I_Po];
      q.RPIo = I[STAGE_TAIL_I_RPIo]; q.phase_rows = I[STAGE_TAIL_I_phase_rows]; q.CS = I[STAGE_TAIL_I_CS];
      VQA_REQUIRE(C % 8 == 0 && q.C8 >= 1 && kTailThreads % q.C8 == 0, VQA_E_INVALID, "stage_tail: C/8 must divide 512");
      VQA_REQUIRE(q.CS == 1 || q.CS == 2 || q.CS == 4 || q.CS == 8, VQA_E_INVALID, "stage_tail: cluster size must be 1, 2, 4 or 8");
      VQA_REQUIRE(q.H % q.CS == 0 && (!q.mode || (q.H / q.CS) % 2 == 0) && (!q.mode || q.W % 2 == 0), VQA_E_INVALID,
                  "stage_tail: rows per CTA must be whole (and even for the phase split)");
      VQA_REQUIRE(q.wconv == nullptr || q.CS == 1, VQA_E_INVALID, "stage_tail: spatial attention needs the whole image (CS = 1)");
      VQA_REQUIRE(q.R <= 256 && (q.w1 == nullptr) == (q.w2 == nullptr), VQA_E_INVALID, "stage_tail: SE hidden width > 256");
      VQA_REQUIRE(q.Po > 0 && q.RPIo % q.Po == 0, VQA_E_INVALID, "stage_tail: bad destination grid");
      const int NP = q.H / q.CS * q.W, lanes = kTailThreads / q.C8;
      const int part_rows = lanes / (q.C8 < 32 ? 32 / q.C8 : 1);
      const int red_rows = part_rows > 8 ? part_rows / 2 : part_rows;
      VQA_REQUIRE(q.C8 >= 32 || 32 % q.C8 == 0, VQA_E_INVALID, "stage_tail: C/8 must divide 32 or be a multiple of it");
      VQA_REQUIRE(q.wconv == nullptr || 2 * NP <= red_rows * C, VQA_E_INVALID, "stage_tail: spatial maps do not fit the scratch area");
      VQA_REQUIRE(q.ks >= 0 && 2 * q.ks * q.ks <= 128, VQA_E_INVALID, "stage_tail: spatial kernel too large");
      const bool f32 = I[STAGE_TAIL_I_f32] != 0;
      q.sums = PTR(const float*, STAGE_TAIL_P_sums);
      if (I[STAGE_TAIL_I_split] > 0) {   // streaming form: slab sums from the producer, no spatial attention, bf16
        SeStreamParams sp;
        sp.src = q.src; sp.dst = q.dst; sp.sums = q.sums; sp.w1 = q.w1; sp.w2 = q.w2; sp.scale_out = q.scale_out;
        sp.B = I[STAGE_TAIL_I_B]; sp.C8 = q.C8; sp.H = q.H; sp.W = q.W; sp.P = q.P; sp.RPI = q.RPI; sp.R = q.R; sp.mode = q.mode;
        sp.Po = q.Po; sp.RPIo = q.RPIo; sp.phase_rows = q.phase_rows; sp.split = I[STAGE_TAIL_I_split];
        VQA_REQUIRE(!f32 && q.wconv == nullptr && q.sums != nullptr && q.w1 != nullptr, VQA_E_INVALID,
                    "stage_tail: the streaming form needs slab sums, SE weights, bf16 data and no spatial attention");
        VQA_REQUIRE(kStreamThreads % q.C8 == 0 && C <= kStreamMaxC && q.R <= 64, VQA_E_INVALID, "stage_tail: streaming form: C/8 must divide 256, C <= 512");
        VQA_REQUIRE(sp.split >= 1 && q.H % sp.split == 0 && (!q.mode || ((q.H / sp.split) % 2 == 0 && q.W % 2 == 0)), VQA_E_INVALID,
                    "stage_tail: rows per CTA must be whole (and even for the phase split)");
        VQA_CUDA_OK(vqa_launch(se_stream_kernel, dim3(sp.B * sp.split), dim3(kStreamThreads), 0, st, sp));
        VQA_LAUNCH_OK("se_stream_kernel");
        return VQA_OK;
      }
      {   // two-pass form: SE-only stages in bf16 (rows re-read from L2 instead of staged in shared memory)
        static const bool two_pass_on = std::getenv("VQA_TAIL_TWO_PASS") == nullptr || std::atoi(std::getenv("VQA_TAIL_TWO_PASS")) != 0;
        if (two_pass_on && !f32 && q.wconv == nullptr && q.w1 != nullptr && kTwoPassThreads % q.C8 == 0 && C <= 512 && q.R <= 64) {
          VQA_CUDA_OK(vqa_launch_cluster(se_two_pass_kernel, dim3(I[STAGE_TAIL_I_B] * q.CS), dim3(kTwoPassThreads), 0, st, q.CS, q));
          VQA_LAUNCH_OK("se_two_pass_kernel");
          return VQA_OK;
        }
      }
      const size_t smem = static_cast<size_t>(NP) * C * (f32 ? 4 : 2) + sizeof(float) * (static_cast<size_t>(red_rows) * C + 2 * C + 256 + NP + 128);
      VQA_REQUIRE(smem <= 227 * 1024, VQA_E_INVALID, "stage_tail: rows per CTA exceed shared memory (raise CS)");
      static bool attr_set[kMaxDevices] = {};   // per device: the attribute belongs to the device's context
      int dev = 0;
      VQA_CUDA_OK(cudaGetDevice(&dev));
      if (dev < 0 || dev >= kMaxDevices || !attr_set[dev]) {
        VQA_CUDA_OK(cudaFuncSetAttribute(reinterpret_cast<const void*>(&stage_tail_kernel<false>),
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        VQA_CUDA_OK(cudaFuncSetAttribute(reinterpret_cast<const void*>(&stage_tail_kernel<true>),
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        if (dev >= 0 && dev < kMaxDevices) attr_set[dev] = true;
      }
      if (f32) {
        VQA_CUDA_OK(vqa_launch_cluster(stage_tail_kernel<true>, dim3(I[STAGE_TAIL_I_B] * q.CS), dim3(kTailThreads), smem, st, q.CS, q));
      } else {
        VQA_CUDA_OK(vqa_launch_cluster(stage_tail_kernel<false>, dim3(I[STAGE_TAIL_I_B] * q.CS), dim3(kTailThreads), smem, st, q.CS, q));
      }
      VQA_LAUNCH_OK("stage_tail_kernel");
      return VQA_OK;
    }
    case VQA_OP_SPLIT_TF32: {
      const int M = I[SPLIT_TF32_I_M], K = I[SPLIT_TF32_I_K], ld = I[SPLIT_TF32_I_ld_src];
      const float* src = PTR(const float*, SPLIT_TF32_P_src);
      VQA_REQUIRE(K % 4 == 0 && ld % 4 == 0 && (reinterpret_cast<uintptr_t>(src) & 15) == 0, VQA_E_ALIGN,
                  "split_tf32: K and the leading dimension must be multiples of 4");
      VQA_CUDA_OK(vqa_launch(split_tf32_kernel, dim3(blocks_for(static_cast<long long>(M) * (K / 4), 256)), dim3(256), 0, st,
                             src, PTR(float*, SPLIT_TF32_P_dst), M, K / 4, ld));
      VQA_LAUNCH_OK("split_tf32_kernel");
      return VQA_OK;
    }
    case VQA_OP_COPY_ROWS: {
      const long long total = static_cast<long long>(I[COPY_ROWS_I_rows]) * I[COPY_ROWS_I_cols];
      VQA_CUDA_OK(vqa_launch(copy_rows_kernel, dim3(blocks_for(total, 256)), dim3(256), 0, st, PTR(const float*, COPY_ROWS_P_src), PTR(float*, COPY_ROWS_P_dst),
                                                               I[COPY_ROWS_I_rows], I[COPY_ROWS_I_cols],
                                                               I[COPY_ROWS_I_ld_src], I[COPY_ROWS_I_ld_dst]));
      VQA_LAUNCH_OK("copy_rows_kernel");
      return VQA_OK;
    }
    case VQA_OP_MASK_PREP: {
      const int n = I[MASK_PREP_I_B] * I[MASK_PREP_I_L];
      const void* src = PTR(const void*, MASK_PREP_P_src);
      VQA_REQUIRE(src != nullptr || I[MASK_PREP_I_dtype] == 0, VQA_E_INVALID, "mask_prep: null mask");
      VQA_CUDA_OK(vqa_launch(mask_prep_kernel, dim3(blocks_for(n, 256)), dim3(256), 0, st, src, PTR(int*, MASK_PREP_P_dst),
                             PTR(float*, MASK_PREP_P_dstf), n, I[MASK_PREP_I_dtype]));
      VQA_LAUNCH_OK("mask_prep_kernel");
      return VQA_OK;
    }
    case VQA_OP_EMBED: {
      const int T = I[EMBED_I_B] * I[EMBED_I_L], D4 = I[EMBED_I_D] / 4;
      const long long* ids = PTR(const long long*, EMBED_P_ids);
      VQA_REQUIRE(ids != nullptr, VQA_E_INVALID, "embed: null token ids");
      if (op.p[EMBED_P_gamma] != 0) {   // + first LayerNorm (+ mask normalisation) in the same launch
        VQA_REQUIRE(I[EMBED_I_D] == 256 && op.p[EMBED_P_beta] != 0 && op.p[EMBED_P_ln_dst] != 0, VQA_E_INVALID,
                    "embed: the fused LayerNorm needs D = 256, beta and an output");
        const void* msrc = PTR(const void*, EMBED_P_mask_src);
        int* mdst = PTR(int*, EMBED_P_mask_dst);
        VQA_REQUIRE(mdst == nullptr || msrc != nullptr || I[EMBED_I_mask_dtype] == 0, VQA_E_INVALID, "embed: null mask");
        VQA_CUDA_OK(vqa_launch(embed_ln_kernel, dim3(blocks_for(T, 8)), dim3(256), 0, st, ids, PTR(const float*, EMBED_P_table),
                               PTR(const float*, EMBED_P_pe), PTR(float*, EMBED_P_dst), PTR(const float*, EMBED_P_gamma),
                               PTR(const float*, EMBED_P_beta), PTR(float*, EMBED_P_ln_dst), T, I[EMBED_I_L], I[EMBED_I_V],
                               I[EMBED_I_round_tf32], op.f[EMBED_F_eps], msrc, mdst, PTR(float*, EMBED_P_mask_dstf),
                               I[EMBED_I_mask_dtype]));
        VQA_LAUNCH_OK("embed_ln_kernel");
        return VQA_OK;
      }
      VQA_CUDA_OK(vqa_launch(embed_kernel, dim3(blocks_for(static_cast<long long>(T) * D4, 256)), dim3(256), 0, st, 
          ids, PTR(const float4*, EMBED_P_table), PTR(const float4*, EMBED_P_pe), PTR(float4*, EMBED_P_dst), T,
          I[EMBED_I_L], D4, I[EMBED_I_V]));
      VQA_LAUNCH_OK("embed_kernel");
      return VQA_OK;
    }
    case VQA_OP_LAYERNORM: {
      VQA_REQUIRE(I[LAYERNORM_I_D] == 256, VQA_E_INVALID, "layernorm: D must be 256");
      const int rows = I[LAYERNORM_I_rows];
      LnExtra ex;
      ex.gamma2 = PTR(const float*, LAYERNORM_P_gamma2); ex.beta2 = PTR(const float*, LAYERNORM_P_beta2);
      ex.dst2 = PTR(float*, LAYERNORM_P_dst2); ex.rnd2 = I[LAYERNORM_I_rnd2];
      ex.gamma3 = PTR(const float*, LAYERNORM_P_gamma3); ex.beta3 = PTR(const float*, LAYERNORM_P_beta3);
      ex.dst3 = PTR(float*, LAYERNORM_P_dst3); ex.rnd3 = I[LAYERNORM_I_rnd3];
      VQA_REQUIRE((ex.gamma2 == nullptr || (ex.beta2 != nullptr && ex.dst2 != nullptr)) &&
                      (ex.gamma3 == nullptr || (ex.beta3 != nullptr && ex.dst3 != nullptr)),
                  VQA_E_INVALID, "layernorm: a chained LayerNorm needs gamma, beta and an output");
      VQA_CUDA_OK(vqa_launch(layernorm256_kernel, dim3(blocks_for(rows, 8)), dim3(256), 0, st, 
          PTR(const float*, LAYERNORM_P_src), PTR(const float*, LAYERNORM_P_gamma), PTR(const float*, LAYERNORM_P_beta),
          PTR(float*, LAYERNORM_P_dst), PTR(const float*, LAYERNORM_P_pos), rows, I[LAYERNORM_I_ld_src],
          I[LAYERNORM_I_mode], I[LAYERNORM_I_round_tf32], I[LAYERNORM_I_S], I[LAYERNORM_I_Pg], I[LAYERNORM_I_RPIg],
          op.f[LAYERNORM_F_eps], ex));
      VQA_LAUNCH_OK("layernorm256_kernel");
      return VQA_OK;
    }
    case VQA_OP_SELF_ATTN: {
      const int L = I[SELF_ATTN_I_L], H = I[SELF_ATTN_I_H], B = I[SELF_ATTN_I_B];
      VQA_REQUIRE(L >= 1 && L <= 64 && I[SELF_ATTN_I_hd] == kHd, VQA_E_INVALID, "self_attn: L<=64, head_dim=32");
      const float* qkv = PTR(const float*, SELF_ATTN_P_qkv);
      const int D = H * kHd, ld = I[SELF_ATTN_I_ld_qkv];
      VQA_REQUIRE(ld % 4 == 0 && (reinterpret_cast<uintptr_t>(qkv) & 15) == 0, VQA_E_ALIGN, "self_attn: qkv alignment");
      VQA_REQUIRE((reinterpret_cast<uintptr_t>(PTR(float*, SELF_ATTN_P_out)) & 15) == 0, VQA_E_ALIGN, "self_attn: out alignment");
      return launch_attn(qkv, qkv + D, qkv + 2 * D, PTR(const int*, SELF_ATTN_P_mask), PTR(float*, SELF_ATTN_P_out), nullptr, B,
                         H, L, L, ld, ld, I[SELF_ATTN_I_no_round], 1, st);
    }
    case VQA_OP_CROSS_ATTN: {
      const int L = I[CROSS_ATTN_I_L], T = I[CROSS_ATTN_I_T], H = I[CROSS_ATTN_I_H], B = I[CROSS_ATTN_I_B];
      VQA_REQUIRE(L >= 1 && L <= 64 && T >= 1 && T <= 64 && I[CROSS_ATTN_I_hd] == kHd, VQA_E_INVALID,
                  "cross_attn: L<=64, T<=64, head_dim=32");
      const float* kv = PTR(const float*, CROSS_ATTN_P_kv);
      VQA_REQUIRE(I[CROSS_ATTN_I_ld_q] % 4 == 0 && I[CROSS_ATTN_I_ld_kv] % 4 == 0 && I[CROSS_ATTN_I_k_off] % 4 == 0 &&
                      I[CROSS_ATTN_I_v_off] % 4 == 0, VQA_E_ALIGN, "cross_attn: leading dimensions must be multiples of 4");
      return launch_attn(PTR(const float*, CROSS_ATTN_P_q), kv + I[CROSS_ATTN_I_k_off], kv + I[CROSS_ATTN_I_v_off], nullptr,
                         PTR(float*, CROSS_ATTN_P_out), PTR(float*, CROSS_ATTN_P_weights), B, H, L, T, I[CROSS_ATTN_I_ld_q],
                         I[CROSS_ATTN_I_ld_kv], I[CROSS_ATTN_I_no_round], I[CROSS_ATTN_I_q_per_kv] > 0 ? I[CROSS_ATTN_I_q_per_kv] : 1, st);
    }
    case VQA_OP_POOL_GATE_LN: {
      const int phase = I[POOL_GATE_LN_I_phase];
      VQA_REQUIRE(I[POOL_GATE_LN_I_D] == 256, VQA_E_INVALID, "pool_gate_ln: D must be 256");
      VQA_REQUIRE(phase >= 0 && phase <= 2 && (phase != 0 || I[POOL_GATE_LN_I_use_gate] == 0), VQA_E_INVALID,
                  "pool_gate_ln: gating runs as pool -> gate GEMM -> mix (phases 1, 2)");
      VQA_REQUIRE(PTR(float*, POOL_GATE_LN_P_att_pooled) && PTR(float*, POOL_GATE_LN_P_txt_pooled), VQA_E_INVALID,
                  "pool_gate_ln: pooled buffers are required");
      VQA_REQUIRE(phase != 1 || PTR(float*, POOL_GATE_LN_P_cat), VQA_E_INVALID, "pool_gate_ln: phase 1 needs cat");
      VQA_REQUIRE(phase != 2 || PTR(const float*, POOL_GATE_LN_P_pre), VQA_E_INVALID, "pool_gate_ln: phase 2 needs pre");
      VQA_CUDA_OK(vqa_launch(pool_gate_ln_kernel, dim3(I[POOL_GATE_LN_I_B]), dim3(256), 0, st,
          PTR(const float*, POOL_GATE_LN_P_xatt), PTR(const float*, POOL_GATE_LN_P_text),
          PTR(const float*, POOL_GATE_LN_P_mask), PTR(const float*, POOL_GATE_LN_P_pre),
          PTR(const float*, POOL_GATE_LN_P_gamma), PTR(const float*, POOL_GATE_LN_P_beta),
          PTR(float*, POOL_GATE_LN_P_fused), PTR(float*, POOL_GATE_LN_P_att_pooled),
          PTR(float*, POOL_GATE_LN_P_txt_pooled), PTR(float*, POOL_GATE_LN_P_cat), I[POOL_GATE_LN_I_L], phase,
          I[POOL_GATE_LN_I_no_round], op.f[POOL_GATE_LN_F_eps]));
      VQA_LAUNCH_OK("pool_gate_ln_kernel");
      return VQA_OK;
    }
    case VQA_OP_SOFTMAX_TOPK: {
      const int N = I[SOFTMAX_TOPK_I_N], k = I[SOFTMAX_TOPK_I_k];
      VQA_REQUIRE(k >= 1 && k <= 128 && k <= N && N <= 10000, VQA_E_INVALID, "softmax_topk: 1<=k<=min(128, N), N<=10000");
      VQA_CUDA_OK(vqa_launch(softmax_topk_kernel, dim3(I[SOFTMAX_TOPK_I_B]), dim3(256), (N + 64 + (N + 31) / 32) * sizeof(float), st, 
          PTR(const float*, SOFTMAX_TOPK_P_logits), PTR(long long*, SOFTMAX_TOPK_P_idx),
          PTR(float*, SOFTMAX_TOPK_P_probs), N, k, I[SOFTMAX_TOPK_I_ld]));
      VQA_LAUNCH_OK("softmax_topk_kernel");
      return VQA_OK;
    }
    default:
      vqa_set_error("unknown op kind " + std::to_string(op.kind));
      return VQA_E_INVALID;
  }
}

const char* misc_kernel_name(int kind) {
  switch (kind) {
    case VQA_OP_INGEST: return "ingest_kernel";
    case VQA_OP_MAXPOOL: return "maxpool_kernel";
    case VQA_OP_SE_SQUEEZE: return "se_squeeze_kernel";
    case VQA_OP_SE_EXCITE: return "se_excite_kernel";
    case VQA_OP_SPATIAL_MAP: return "spatial_map_kernel";
    case VQA_OP_SCALE_RELAYOUT: return "scale_relayout_kernel";
    case VQA_OP_GRID_TO_NCHW: return "grid_to_nchw_kernel";
    case VQA_OP_MASK_PREP: return "mask_prep_kernel";
    case VQA_OP_COPY_ROWS: return "copy_rows_kernel";
    case VQA_OP_SPLIT_TF32: return "split_tf32_kernel";
    case VQA_OP_STAGE_TAIL: return "stage_tail_kernel";
    case VQA_OP_EMBED: return "embed_kernel";
    case VQA_OP_LAYERNORM: return "layernorm256_kernel";
    case VQA_OP_SELF_ATTN: return "attn_mma_kernel(self)";
    case VQA_OP_CROSS_ATTN: return "attn_mma_kernel(cross)";
    case VQA_OP_POOL_GATE_LN: return "pool_gate_ln_kernel";
    case VQA_OP_SOFTMAX_TOPK: return "softmax_topk_kernel";
    default: return "?";
  }
}
