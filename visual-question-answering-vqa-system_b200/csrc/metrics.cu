// Fused top-1 / top-k accuracy accumulation on the device (SURVEY 8(f) row f4).
//
// Replaces the per-batch host work of the reference's evaluation loop: VQAAccuracy.update (utils/metrics.py:56-105)
// takes argmax and topk(5) of the logits, moves predictions and targets to the CPU and calls .item() twice per batch
// (training/evaluate.py:77-106, training/train.py:229-264).  Here one kernel per batch ranks the target's logit inside
// its row and adds to three 64-bit counters that stay in HBM; the host reads them once, in compute().
//
// rank(row) = #{ j : v[j] ranks before v[t] }   (t = target; rank_before: NaN > +inf > finite > -inf, ties go to the lower
// index, the order torch.argmax / torch.topk pick), so  top-1 correct <=> rank == 0  and  top-k correct <=> rank < k, and
// the predicted index is torch.argmax's (the first NaN of a row that has one).  A target outside
// [0, N) (AnswerVocabulary.encode returns -1 for unknown answers, data/build_vocab.py:205-218) is never correct and
// still counts in `total`, exactly as in the reference.  One warp per row; HBM-bound: the logits are read once
// (4 N bytes per row).
#include "common.cuh"

namespace {

constexpr int kWarpsPerBlock = 8;

__global__ void __launch_bounds__(kWarpsPerBlock * 32)
accuracy_kernel(const float* __restrict__ logits, int ld, int N, const long long* __restrict__ pred_in,
                const long long* __restrict__ targets, int B, int k, unsigned long long* __restrict__ counters,
                long long* __restrict__ pred_out, int* __restrict__ rank_out) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ unsigned int s_top1, s_topk;
  if (threadIdx.x == 0) { s_top1 = 0u; s_topk = 0u; }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  // one warp per row, one short-lived block per 8 rows: thousands of blocks in flight hide the dependent
  // target -> v[target] loads at the head of every row (a grid-stride variant sized to the SM count measured 3.3 TB/s
  // against 4.3-5.1 TB/s for this form)
  const int row = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (row < B) {
    const long long t = targets[row];
    if (logits == nullptr) {
      // predictions are indices already ([B] form of VQAAccuracy.update): top-1 only
      const long long p = pred_in[row];
      if (lane == 0) {
        if (p == t) atomicAdd(&s_top1, 1u);
        if (pred_out) pred_out[row] = p;
        if (rank_out) rank_out[row] = (p == t) ? 0 : N;
      }
    } else {
      const float* v = logits + static_cast<size_t>(row) * ld;
      const bool valid = t >= 0 && t < N;
      const float tv = valid ? v[t] : INFINITY;
      const int ti = valid ? static_cast<int>(t) : -1;
      int above = 0;
      float best = -INFINITY, special = 0.f;
      int bi = 0x7fffffff;
      // the streaming pass compares as for finite rows and only notes whether the row holds a NaN or an infinity
      // (x * 0 is NaN then): comparing every element with rank_before here halved the achieved bandwidth
      auto visit = [&](float x, int j) {
        above += (x > tv || (x == tv && j < ti)) ? 1 : 0;
        if (x > best || (x == best && j < bi)) { best = x; bi = j; }
        special = fmaf(x, 0.f, special);
      };
      if (((reinterpret_cast<uintptr_t>(v) | (static_cast<uintptr_t>(ld) * 4)) & 15) == 0) {
        // 16-byte loads (row pitch and base aligned): 512 bytes per warp instruction, two in flight per lane
        const float4* v4 = reinterpret_cast<const float4*>(v);
        const int n4 = N >> 2;
        int q = lane;
        for (; q + 32 < n4; q += 64) {
          const float4 a = __ldg(v4 + q), b = __ldg(v4 + q + 32);
          visit(a.x, 4 * q); visit(a.y, 4 * q + 1); visit(a.z, 4 * q + 2); visit(a.w, 4 * q + 3);
          visit(b.x, 4 * q + 128); visit(b.y, 4 * q + 129); visit(b.z, 4 * q + 130); visit(b.w, 4 * q + 131);
        }
        for (; q < n4; q += 32) {
          const float4 a = __ldg(v4 + q);
          visit(a.x, 4 * q); visit(a.y, 4 * q + 1); visit(a.z, 4 * q + 2); visit(a.w, 4 * q + 3);
        }
        for (int j = (n4 << 2) + lane; j < N; j += 32) visit(v[j], j);
      } else {
#pragma unroll 8
        for (int j = lane; j < N; j += 32) visit(v[j], j);
      }
      if (__any_sync(0xffffffffu, special != special)) {
        // a NaN or an infinity in the row: recount it in rank_before's order (the row is read a second time)
        above = 0;
        best = -INFINITY;
        bi = 0x7fffffff;
        for (int j = lane; j < N; j += 32) {
          const float x = v[j];
          above += rank_before(x, j, tv, ti) ? 1 : 0;
          if (rank_before(x, j, best, bi)) { best = x; bi = j; }
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        above += __shfl_xor_sync(0xffffffffu, above, o);
        const float ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (rank_before(ob, oi, best, bi)) { best = ob; bi = oi; }
      }
      if (lane == 0) {
        if (valid && above == 0) atomicAdd(&s_top1, 1u);
        if (valid && above < k) atomicAdd(&s_topk, 1u);
        if (pred_out) pred_out[row] = bi;
        if (rank_out) rank_out[row] = valid ? above : N;
      }
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (s_top1) atomicAdd(&counters[0], static_cast<unsigned long long>(s_top1));
    if (s_topk) atomicAdd(&counters[1], static_cast<unsigned long long>(s_topk));
    if (blockIdx.x == 0) atomicAdd(&counters[2], static_cast<unsigned long long>(B));
  }
}

}  // namespace

extern "C" int vqa_accuracy_update(const float* logits, int32_t ld, int32_t num_classes, const int64_t* pred_in,
                                   const int64_t* targets, int32_t batch, int32_t k, uint64_t* counters,
                                   int64_t* pred_out, int32_t* rank_out, void* stream) {
  VQA_REQUIRE(targets != nullptr && counters != nullptr, VQA_E_INVALID, "accuracy: null targets / counters");
  VQA_REQUIRE((logits != nullptr) != (pred_in != nullptr), VQA_E_INVALID,
              "accuracy: give either logits [B, N] or predicted indices [B]");
  VQA_REQUIRE(batch >= 0 && num_classes >= 1 && k >= 1, VQA_E_INVALID, "accuracy: bad batch / num_classes / k");
  VQA_REQUIRE(logits == nullptr || ld >= num_classes, VQA_E_INVALID, "accuracy: ld < num_classes");
  VQA_REQUIRE((reinterpret_cast<uintptr_t>(counters) & 7) == 0, VQA_E_ALIGN, "accuracy: counters must be 8-byte aligned");
  if (batch == 0) return VQA_OK;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  VQA_CUDA_OK(vqa_launch(accuracy_kernel, dim3((batch + kWarpsPerBlock - 1) / kWarpsPerBlock), dim3(kWarpsPerBlock * 32), 0,
                         st, logits, static_cast<int>(ld), static_cast<int>(num_classes),
                         reinterpret_cast<const long long*>(pred_in), reinterpret_cast<const long long*>(targets),
                         static_cast<int>(batch), static_cast<int>(k), reinterpret_cast<unsigned long long*>(counters),
                         reinterpret_cast<long long*>(pred_out), reinterpret_cast<int*>(rank_out)));
  VQA_LAUNCH_OK("accuracy_kernel");
  return VQA_OK;
}
