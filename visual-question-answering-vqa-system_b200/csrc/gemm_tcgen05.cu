// Tap-shifted GEMM on tcgen05 / TMEM fed by TMA  (VQA_OP_GEMM), persistent and warp-specialised.
//
// One kernel covers every Conv2d(+BN folded)(+ReLU)(+residual) of the backbone
// (reference models/cnn_backbone.py:164-197, 349-352) and every nn.Linear of the text encoder,
// fusion module and answer head: out[M,N] = sum_g sum_t A_g[m + delta_g - halo + rel_t, :] * W_t^T.
//
// Data layout (see program.py): A is a 2-D K-major tensor (rows = padded-flat pixels or tokens,
// 128-byte K chunks), W is [Npad, Ktot] K-major.  Per K chunk the producer warp TMA-loads ONE
// window of A rows (tile rows + halo on both sides, SWIZZLE_128B) and the MMA thread issues one
// UMMA set per tap whose A descriptor starts `rel` rows into that window -- a 3x3 convolution
// re-uses each input row 9 times out of shared memory instead of re-fetching it from L2.
// (Measured on B200: the UMMA SWIZZLE_128B pattern is a function of the absolute shared-memory
// address, so a start address offset by whole 128-byte rows needs no base_offset correction.)
//
// CTA = 10 warps, one CTA per SM, looping over output tiles (static round-robin):
//   warp 0      TMA producer: A-window ring + weight ring (or all weights resident when they fit)
//   warp 1      MMA issuer: one thread issues tcgen05.mma; tcgen05.commit frees ring slots
//   warps 2..9  epilogue: TMEM -> registers -> bias / TMA-loaded residual / ReLU / pad-mask -> swizzled staging ->
//               TMA store; two warps per TMEM lane quadrant, each taking half of the tile's columns
//               (EPI 4, the stem: ReLU -> shared-memory conv tile -> 3x3/2 max-pool -> global)
// Accumulators are double-buffered in TMEM (when 2*MT*BN <= 512 columns) so the epilogue of tile
// i overlaps the MMAs of tile i+1.  PAIR = true runs two CTAs of a cluster as one cta_group::2 unit
// (256-row UMMA, half of every weight tile per CTA).  Every launch carries the programmatic-dependent-
// launch attribute: prologue and weight prefetch run before griddepcontrol.wait.
#include <cstdio>
#include <type_traits>

#include <cstdlib>

#include "common.cuh"

namespace {

constexpr int kEpiWarps = 8;
constexpr int kThreads = 32 * (2 + kEpiWarps);   // producer, MMA issuer, 8 epilogue warps
constexpr int kSfEpiWarps = 16;                  // shift-fused kernels: 16 epilogue warps (their epilogue is issue-bound)
constexpr int kSfThreads = 32 * (2 + kSfEpiWarps);
constexpr int kMaxEpiWarps = 16;
constexpr int kMaxASlots = 8;
constexpr int kMaxBSlots = 12;

struct GemmParams {
  int M, N;
  int MT;            // 128-row sub-tiles per CTA tile (1 or 2); mirrors the kernel's template MT
  int halo;          // window rows before the tile (halo_hi rows after it)
  int box_rows;      // TMA box rows for A
  int nboxes;        // boxes per window (1..3)
  int row_bytes;     // K-chunk width: 128 (SWIZZLE_128B, 4 MMAs per chunk) or 32 (SWIZZLE_32B, 1 MMA per chunk)
  int a_tx_bytes;    // bytes one window load delivers (nboxes * box_rows * row_bytes)
  uint32_t desc_hi;  // high word of the UMMA shared-memory descriptor (SBO, version, swizzle mode)
  int a_slots, b_slots;
  int a_slot_bytes, b_slot_bytes;
  int b_resident;    // all weight chunks of the N tile stay in shared memory for the CTA's lifetime
  int k_chunks;      // Ktot / chunk_elems
  int acc_stages;    // TMEM accumulator double buffering (1 or 2)
  int win_per_tile;  // A windows one tile consumes (sum of chunks over groups)
  int steps_per_tile;// weight tiles one tile consumes (sum of chunks*taps over groups)
  int m_tiles, n_tiles;   // tiles a CTA (or, in pair mode, a CTA pair) walks: m_tiles counts pairs of m tiles then
  int m_tiles_cta;        // real number of per-CTA m tiles (pair mode: the last pair may hold a phantom tile)
  int ngroups;
  int chunk_elems;   // 64 (bf16) / 32 (tf32)
  int is_tf32;
  uint32_t idesc;
  int g_map[VQA_MAX_GROUPS], g_delta[VQA_MAX_GROUPS], g_acol[VQA_MAX_GROUPS], g_chunks[VQA_MAX_GROUPS];
  int g_ntaps[VQA_MAX_GROUPS], g_kbase[VQA_MAX_GROUPS], g_tap0[VQA_MAX_GROUPS];
  int g_q0[VQA_MAX_GROUPS];   // g_kbase / chunk_elems (first weight chunk of the group)
  int tap_rel[VQA_MAX_TAPS];
  // epilogue
  void* out;
  const float* bias;
  const void* res;
  int ldo, ldr, out_dtype, res_dtype;
  int relu, round_tf32, mask_en, mP, mRPI, mH, mW;
  int out_f16;       // 16-bit outputs are fp16 instead of bf16 (operands of the fp16 tail GEMMs)
  // programmatic dependent launch trigger: 0 = right after the prologue, 1 = when this CTA's producer starts its LAST tile
  // (dependents' CTAs spin at griddepcontrol.wait on the SMs they get: triggering late leaves the SMs that finish early to
  // the other compute lanes' kernels instead)
  int pdl_late;
  // strided M tiling (fused stem + max-pool): tile t starts at (t / tiles_per_img) * img_rows +
  // (t % tiles_per_img) * tile_stride + tile_row0 instead of t * 128 * MT  (tiles_per_img = 0: linear)
  int tiles_per_img, tile_stride, tile_row0, img_rows;
  // fused 3x3/2 max-pool epilogue (EPI 4): conv grid pitch / width, pooled grid geometry
  int pool_P, pool_W, pool_Wo, pool_Ho, pool_Po, pool_rpio;
  // shift-fused form (template SF > 1): the accumulator holds SF column blocks of BN; out[r] = sum_j acc[r + j*sf_step][j*BN + n]
  int sf_step;
  // pad mask without integer division: n / d = umulhi(n, magic) >> shift for every n < 2^31 (checked on the host)
  uint32_t rpi_magic, rpi_shift, mp_magic, mp_shift;
  // optional per-slab column sums of the stored values (SE squeeze partial sums, models/attention_modules.py:116):
  // sums[(row / 32) * ld_sums + n] = sum over the 32 rows of that slab of out[row, n] (fp32, before the 16-bit rounding)
  float* sums;
  int ld_sums;
  // fused softmax + top-k of the output rows (EPI 6: the answer head's last Linear, models/vqa_model.py:336-337):
  // every epilogue thread keeps the running max / exp-sum / k best of its row over the columns it drains and writes them as
  // partial (row, n_tile, column half); the CTA that finishes the last N tile of an M tile (atomic counter) merges them
  long long* topk_idx;   // [M, topk_k] winners, best first (rank_before: ties to the lower index, NaN first like torch.topk)
  float* topk_probs;     // [M, topk_k] softmax probabilities of the winners
  float* topk_part;      // [M, 2 * n_tiles, 2 + 2 * kTopKMax] scratch
  int* topk_cnt;         // [m_tiles] arrival counters (zero between launches: the merging CTA resets its counter)
  int topk_k;
  long long* dbg;    // optional: 16 clock64() timestamps of CTA 0 (profiling aid, nullptr in production)
};

// Column sums of a 32 x 32 block held one row per lane: after 31 shuffles lane l holds sum over lanes of s[l] (fixed
// order, so the result is deterministic).  Step with offset o: the half of the warp with bit o set keeps the upper o
// columns and receives the partner's upper o columns, the other half the lower ones.  Destroys s.
__device__ __forceinline__ float warp_colsum32(float (&s)[32], int lane) {
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) {
    const bool up = (lane & o) != 0;
#pragma unroll
    for (int k = 0; k < o; ++k) {
      const float send = up ? s[k] : s[k + o];
      const float keep = up ? s[k + o] : s[k];
      s[k] = keep + __shfl_xor_sync(0xffffffffu, send, o);
    }
  }
  return s[0];
}

__device__ __forceinline__ int tile_m0(const GemmParams& p, int tile_m, int mt) {
  if (p.tiles_per_img == 0) return tile_m * 128 * mt;
  const int img = tile_m / p.tiles_per_img;
  return img * p.img_rows + (tile_m - img * p.tiles_per_img) * p.tile_stride + p.tile_row0;
}

// rem = row % rpi, then (rem / P, rem % P) against (H, W): true for an in-image position of the padded-flat grid
__device__ __forceinline__ bool grid_pixel(const GemmParams& p, int row) {
  const uint32_t n = static_cast<uint32_t>(row);
  const uint32_t rem = n - (__umulhi(n, p.rpi_magic) >> p.rpi_shift) * static_cast<uint32_t>(p.mRPI);
  const uint32_t h = __umulhi(rem, p.mp_magic) >> p.mp_shift;
  return h < static_cast<uint32_t>(p.mH) && rem - h * static_cast<uint32_t>(p.mP) < static_cast<uint32_t>(p.mW);
}

constexpr int kTopKMax = 8;             // fused top-k epilogue: winners kept per thread (larger k: softmax_topk_kernel)
constexpr int kTopKRec = 4 + 2 * kTopKMax;   // floats per partial record (80 bytes): max, exp-sum, 2 pad, keys, indices
// (key, index) beats (key', index') when it ranks before it (rank_before); the list stays sorted best first
__device__ __forceinline__ void topk_insert(float (&tv)[kTopKMax], int (&ti)[kTopKMax], float key, int idx) {
  if (!rank_before(key, idx, tv[kTopKMax - 1], ti[kTopKMax - 1])) return;
#pragma unroll
  for (int j = kTopKMax - 1; j >= 0; --j) {
    const bool better = rank_before(key, idx, tv[j], ti[j]);
    if (better) {
      if (j + 1 < kTopKMax) { tv[j + 1] = tv[j]; ti[j + 1] = ti[j]; }
      tv[j] = key;
      ti[j] = idx;
    }
  }
}

#define VQA_DBG(slot)                                                         \
  do {                                                                        \
    if (p.dbg && blockIdx.x == 0 && lane == 0) p.dbg[slot] = clock64();       \
  } while (0)

// ---- epilogue --------------------------------------------------------------------------------
// The accumulator comes out of TMEM one row per lane.  Writing rows straight to global memory
// makes every 16-byte store of a warp touch 32 different 128-byte lines (measured: 14k cycles for
// a 128x256 fp32 tile), so all global traffic of the epilogue goes through TMA instead: each
// epilogue warp finishes its 32x32 chunk in the row-per-lane domain (bias from a shared-memory
// table, residual from a TMA-loaded box, ReLU / pad mask / rounding), writes the result as a
// swizzled box into its private staging slot and one lane issues a TMA store, which also clips
// the M and N edges.  The residual box of the NEXT chunk is in flight while the current one is
// processed.  Slots are 32 rows x 64 B (bf16, SWIZZLE_64B) or 32 rows x 128 B (fp32, SWIZZLE_128B).
constexpr int kBiasTable = 2048;        // floats: bias of every N tile of the launch (wider layers read it from global)
constexpr int kXchgRows = 4;            // shift-fused epilogue: accumulator rows a warp publishes for the warp above it
constexpr int kXchgBytes = 2 * kSfEpiWarps * kXchgRows * 16 * 4; // double-buffered, one slot of 16-column rows per warp
constexpr int kPoolTileBytes = 384 * 128;

__host__ __device__ constexpr int epi_stage_bytes(int epi, int sf = 1) {
  if (sf > 1) return kSfEpiWarps * 2048 * ((epi & 1) ? 2 : 1);   // shift-fused: 32 rows x 32 bf16 channels per warp
  return epi == 4 ? kPoolTileBytes : kEpiWarps * ((epi < 2 ? 2048 : 4096) * ((epi & 1) ? 2 : 1));
}

// EPI: 0 = bf16 out, no residual | 1 = bf16 out + bf16 residual | 2 = fp32 out, no residual | 3 = fp32 out + fp32 residual
// mbarrier wait that also accumulates the cycles spent waiting (profiling aid, only when dbg is set)
__device__ __forceinline__ void mbar_wait_t(uint64_t* bar, uint32_t parity, bool timed, long long& acc) {
  if (timed) {
    const long long t0 = clock64();
    mbar_wait(bar, parity);
    acc += clock64() - t0;
  } else {
    mbar_wait(bar, parity);
  }
}

// ROW32: K chunks are 32-byte rows (the stem) instead of 128-byte rows.
// PAIR: two CTAs of a cluster share one 256-row UMMA (cta_group::2): each loads its own A windows and HALF of every
// weight tile, the even CTA issues the MMAs for both, each CTA drains its own 128 accumulator rows.
// SF > 1 (shift-fused, MT = 1): every MMA is SF*BN columns wide -- block j of the weight tile holds horizontal tap j --
// and the epilogue adds block j shifted up by j*sf_step accumulator rows (warp shuffles; the rows that come from the
// next 32-row slab go through a small shared-memory exchange).  A 128x64x16 SS-mode MMA is bound by its shared-memory
// operand reads (6 KB per 32 math cycles: 48.6 clk measured, tools/ubench.cu); at N = 192 the same A bytes feed three
// times the math and the MMA runs at its 96-cycle floor.  The last (SF-1)*sf_step rows of a tile have no complete sum:
// tiles advance by 128 - (SF-1)*sf_step rows and the last slab is stored through a shorter box (mapOutLast).
template <int BN, int MT, bool TF32, int EPI, bool ROW32, bool PAIR, int SF = 1>
__global__ void __launch_bounds__(SF > 1 ? kSfThreads : kThreads, 1)
gemm_tap_kernel(const __grid_constant__ CUtensorMap mapA0, const __grid_constant__ CUtensorMap mapA1,
                const __grid_constant__ CUtensorMap mapB, const __grid_constant__ CUtensorMap mapOut,
                const __grid_constant__ CUtensorMap mapRes, const __grid_constant__ CUtensorMap mapOutLast,
                const __grid_constant__ GemmParams p) {
  static_assert(SF == 1 || (MT == 1 && EPI < 2 && !TF32 && !ROW32), "shift-fused tiles: MT = 1, bf16 output");
  constexpr int kAcc = SF * BN;                 // accumulator columns of one 128-row sub-tile
  extern __shared__ uint8_t smem_raw[];
  // SWIZZLE_128B tiles need 1024-byte alignment in the shared window.
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);

  constexpr int kRowBytes = ROW32 ? 32 : 128;   // bytes of one K chunk row
  constexpr int kMmaPerChunk = kRowBytes / 32;  // UMMA K is 32 bytes (16 bf16 / 8 tf32)
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int total_tiles = p.m_tiles * p.n_tiles;
  const uint32_t rank = PAIR ? cluster_rank() : 0u;                  // 0 = leader (issues the MMAs)
  const int walker = PAIR ? static_cast<int>(blockIdx.x >> 1) : static_cast<int>(blockIdx.x);   // tile-sequence id
  const int n_walkers = PAIR ? static_cast<int>(gridDim.x >> 1) : static_cast<int>(gridDim.x);
  // per-CTA m-tile index of a walked tile (pair mode: 2 * pair index + rank; may be a phantom tile >= m_tiles_cta)
  // tile -> (m tile, n tile) without an integer division when there is one N tile (every 64- / 128-channel convolution):
  // the divisions by a runtime value cost ~25 instructions each, several times per tile and warp
  const bool one_ntile = p.n_tiles == 1;
  auto tile_mt = [&](int tile) { return one_ntile ? tile : tile % p.m_tiles; };
  auto tile_nt = [&](int tile) { return one_ntile ? 0 : tile / p.m_tiles; };
  auto cta_mtile = [&](int tile) { return PAIR ? 2 * tile_mt(tile) + static_cast<int>(rank) : tile_mt(tile); };
  const int b_region_slots = p.b_resident ? p.k_chunks : p.b_slots;

  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem_a + p.a_slots * p.a_slot_bytes;
  uint8_t* smem_stage = smem_b + b_region_slots * p.b_slot_bytes;     // 1024-byte aligned (slots are 1 KB multiples)
  float* s_bias = reinterpret_cast<float*>(smem_stage + epi_stage_bytes(EPI, SF));
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_bias + kBiasTable);
  uint64_t* a_full = bars;
  uint64_t* a_empty = a_full + kMaxASlots;
  uint64_t* b_full = a_empty + kMaxASlots;     // b_full[0] doubles as the "all weights landed" barrier
  uint64_t* b_empty = b_full + kMaxBSlots;
  uint64_t* acc_full = b_empty + kMaxBSlots;
  uint64_t* acc_empty = acc_full + 2;
  uint64_t* res_bar = acc_empty + 2;           // one per epilogue warp: "residual box landed"
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(res_bar + kMaxEpiWarps);
  uint32_t* s_rel = tmem_slot + 4;                                   // tap row offsets, pre-shifted for descriptors
  int4* s_grp = reinterpret_cast<int4*>(s_rel + VQA_MAX_TAPS);      // per group {chunks, taps, tap0, q0}
  float* s_xchg = reinterpret_cast<float*>(s_grp + VQA_MAX_GROUPS); // SF > 1 only: boundary rows between epilogue warps

  if (warp == 0) VQA_DBG(0);
  if (p.dbg && blockIdx.x == 0 && threadIdx.x == 0) {
    unsigned long long ns;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(ns));
    p.dbg[22] = static_cast<long long>(ns);
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapA0);
    tma_prefetch_desc(&mapA1);
    tma_prefetch_desc(&mapB);
    if (EPI != 4) tma_prefetch_desc(&mapOut);
    if (SF > 1) tma_prefetch_desc(&mapOutLast);
    if (EPI & 1) tma_prefetch_desc(&mapRes);
  }
  if (warp == 1) {   // barrier / table initialisation spread over the warp's lanes (one thread took ~1k cycles)
    if (lane < kMaxASlots) { mbar_init(&a_full[lane], 1); mbar_init(&a_empty[lane], 1); }
    if (lane < kMaxBSlots) { mbar_init(&b_full[lane], 1); mbar_init(&b_empty[lane], 1); }
    if (lane >= 16 && lane < 18) {   // shift-fused kernels: each accumulator stage is drained by one group of four warps
      mbar_init(&acc_full[lane - 16], 1);
      mbar_init(&acc_empty[lane - 16], kEpiWarps * (PAIR ? 2 : 1));   // SF: 8 of the 16 warps drain each stage
    }
    if (lane < kMaxEpiWarps) mbar_init(&res_bar[lane], 1);
    if (lane < VQA_MAX_TAPS) s_rel[lane] = static_cast<uint32_t>(p.tap_rel[lane]) * (kRowBytes / 16);
    if (lane < VQA_MAX_GROUPS) s_grp[lane] = make_int4(p.g_chunks[lane], p.g_ntaps[lane], p.g_tap0[lane], p.g_q0[lane]);
    __syncwarp();
    if (lane == 0) mbar_fence_init();
  }
  uint32_t tmem_cols = 32;
  while (tmem_cols < static_cast<uint32_t>(kAcc * MT * p.acc_stages)) tmem_cols <<= 1;   // power of two >= 32
  if (warp == 2) {
    if (PAIR) { tmem_alloc_pair(tmem_slot, tmem_cols); tmem_relinquish_pair(); }
    else      { tmem_alloc(tmem_slot, tmem_cols); tmem_relinquish(); }
  }
  tc_fence_before();
  if (PAIR) cluster_sync(); else __syncthreads();       // pair: the peer's barriers must exist before anything signals them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (warp == 0) VQA_DBG(1);
  // Programmatic dependent launch: the next kernel of the stream may start its own prologue now; this one
  // has done everything that does not depend on its predecessors (barriers, TMEM, descriptor prefetch).
  if (warp == 1 && (!p.pdl_late || walker >= total_tiles)) pdl_launch_dependents();

  if (warp == 0) {
    // ===================== TMA producer (whole warp loops, one elected lane issues) =====================
    int as = 0, bs = 0;
    uint32_t aph = 0, bph = 0;
    bool b_loaded = false;
    const bool timed = p.dbg != nullptr && blockIdx.x == 0;
    long long w_aempty = 0, w_bempty = 0;
    // pair mode: every load of either CTA completes on the LEADER's full barrier, which expects both CTAs' bytes
    constexpr uint32_t kTxMul = PAIR ? 2u : 1u;
    const bool expects = !PAIR || rank == 0;
    auto load = [&](void* dst, const CUtensorMap* map, uint64_t* bar, int x, int y) {
      if (PAIR) tma_load_2d_pair(dst, map, bar, x, y); else tma_load_2d(dst, map, bar, x, y);
    };
    for (int tile = walker; tile < total_tiles; tile += n_walkers) {
      if (p.pdl_late && tile + n_walkers >= total_tiles) pdl_launch_dependents();
      const int m0 = tile_m0(p, cta_mtile(tile), MT);
      const int n0 = tile_nt(tile) * kAcc + (PAIR ? static_cast<int>(rank) * (kAcc / 2) : 0);   // pair: this CTA's half of the N tile
      if (p.b_resident && !b_loaded) {   // n_tiles == 1 in this mode: load every weight chunk once
        if (elect_one()) {
          if (expects) mbar_expect_tx(&b_full[0], static_cast<uint32_t>(p.k_chunks * p.b_slot_bytes) * kTxMul);
          for (int q = 0; q < p.k_chunks; ++q)
            load(smem_b + q * p.b_slot_bytes, &mapB, &b_full[0], q * p.chunk_elems, n0);
        }
        __syncwarp();
        b_loaded = true;
      }
      if (tile == walker) pdl_wait();   // weights are constants; the activations are not
      for (int g = 0; g < p.ngroups; ++g) {
        const CUtensorMap* mapA = p.g_map[g] ? &mapA1 : &mapA0;
        const int row0 = m0 + p.g_delta[g] - p.halo;
        for (int c = 0; c < p.g_chunks[g]; ++c) {
          mbar_wait_t(&a_empty[as], aph ^ 1u, timed, w_aempty);
          if (elect_one()) {
            if (expects) mbar_expect_tx(&a_full[as], static_cast<uint32_t>(p.a_tx_bytes) * kTxMul);
            uint8_t* dst = smem_a + as * p.a_slot_bytes;
            const int x = p.g_acol[g] + c * p.chunk_elems;
            for (int b = 0; b < p.nboxes; ++b)
              load(dst + b * p.box_rows * kRowBytes, mapA, &a_full[as], x, row0 + b * p.box_rows);
          }
          __syncwarp();
          if (tile == walker && g == 0 && c == 0) VQA_DBG(2);
          if (++as == p.a_slots) { as = 0; aph ^= 1u; }
          if (!p.b_resident) {
            for (int t = 0; t < p.g_ntaps[g]; ++t) {
              mbar_wait_t(&b_empty[bs], bph ^ 1u, timed, w_bempty);
              if (elect_one()) {
                if (expects) mbar_expect_tx(&b_full[bs], static_cast<uint32_t>(p.b_slot_bytes) * kTxMul);
                const int kcol = p.g_kbase[g] + (t * p.g_chunks[g] + c) * p.chunk_elems;
                load(smem_b + bs * p.b_slot_bytes, &mapB, &b_full[bs], kcol, n0);
              }
              __syncwarp();
              if (++bs == p.b_slots) { bs = 0; bph ^= 1u; }
            }
          }
        }
      }
    }
    if (timed && lane == 0) { p.dbg[16] = w_aempty; p.dbg[17] = w_bempty; }
  } else if (warp == 1) {
    // ===================== MMA issuer: ONE elected thread runs the whole role =====================
    // Inside an elect.sync region ptxas keeps descriptors in uniform registers and emits
    // back-to-back UTCHMMA.  Measured on B200: the cost is the ~200-cycle per-step overhead of a
    // single thread's dependent instruction chain (loop control, tap-table load, address math), not
    // the MMA issue itself (splitting the K slices over two issuer threads changed nothing and made
    // the accumulation order non-deterministic), so the common 9-tap window group is fully unrolled
    // with its tap offsets held in registers and loop-invariant parameters hoisted by hand.
    if ((!PAIR || rank == 0) && elect_one()) {
      const int a_slots = p.a_slots, b_slots = p.b_slots, ngroups = p.ngroups, acc_stages = p.acc_stages;
      const bool resident = p.b_resident != 0;
      const uint32_t a_slot_lo = static_cast<uint32_t>(p.a_slot_bytes) >> 4;
      const uint32_t b_slot_lo = static_cast<uint32_t>(p.b_slot_bytes) >> 4;
      const uint32_t a_base_lo = smem_u32(smem_a) >> 4;
      const uint32_t b_base_lo = smem_u32(smem_b) >> 4;
      const uint32_t idesc = p.idesc;
      const uint64_t kDescHi = static_cast<uint64_t>(p.desc_hi) << 32;
      const bool timed = p.dbg != nullptr && blockIdx.x == 0;
      long long w_accempty = 0, w_afull = 0, w_bfull = 0;
      int as = 0, bs = 0, acc = 0;
      uint32_t aph = 0, bph = 0, accph = 0;
      constexpr int kUnroll = ROW32 ? 16 : 9;   // taps of the unrolled window group (4x4 stem / 3x3 conv)
      uint32_t relu_[kUnroll];                  // group 0's tap offsets in registers
#pragma unroll
      for (int t = 0; t < kUnroll; ++t) relu_[t] = s_rel[t];
      const bool g0_unrolled = p.g_ntaps[0] == kUnroll && p.g_tap0[0] == 0;
      uint32_t d_tile = 0, fresh = 1;

      // one (window, tap) step: kMmaPerChunk*MT MMAs over the K chunk
      auto commit = [&](uint64_t* bar) { if (PAIR) umma_commit_pair(bar); else umma_commit(bar); };   // pair: both CTAs' barriers
      auto issue_step = [&](uint32_t a_lo, uint32_t b_lo) {
#pragma unroll
        for (int sub = 0; sub < MT; ++sub) {
#pragma unroll
          for (int k = 0; k < kMmaPerChunk; ++k) {   // K = 32 bytes per MMA; 32 B >> 4 = 2
            const uint64_t ad = kDescHi | (a_lo + sub * (128 * kRowBytes / 16) + 2 * k);
            const uint64_t bd = kDescHi | (b_lo + 2 * k);
            const uint32_t accum = (k == 0) ? (fresh ^ 1u) : 1u;
            if (PAIR && TF32) umma_tf32_pair(d_tile + sub * kAcc, ad, bd, idesc, accum);
            else if (PAIR)    umma_f16_pair(d_tile + sub * kAcc, ad, bd, idesc, accum);
            else if (TF32)    umma_tf32(d_tile + sub * kAcc, ad, bd, idesc, accum);
            else              umma_f16(d_tile + sub * kAcc, ad, bd, idesc, accum);
          }
        }
        fresh = 0;
      };
      // weight tile of this step: resident chunk q, or the next ring slot (wait / commit around the MMAs)
      auto b_acquire = [&](uint32_t q) -> uint32_t {
        if (resident) return b_base_lo + q * b_slot_lo;
        mbar_wait_t(&b_full[bs], bph, timed, w_bfull);
        tc_fence_after();
        return b_base_lo + bs * b_slot_lo;
      };
      auto b_release = [&]() {
        if (!resident) {
          commit(&b_empty[bs]);            // weight slot is free once these MMAs retire
          if (++bs == b_slots) { bs = 0; bph ^= 1u; }
        }
      };

      if (resident) mbar_wait(&b_full[0], 0);
      for (int tile = walker; tile < total_tiles; tile += n_walkers) {
        mbar_wait_t(&acc_empty[acc], accph ^ 1u, timed, w_accempty);   // epilogue has drained this accumulator stage
        tc_fence_after();
        d_tile = tmem_base + acc * (kAcc * MT);
        fresh = 1;                           // first MMA of each accumulator overwrites, the rest accumulate
        for (int g = 0; g < ngroups; ++g) {
          const int4 grp = s_grp[g];
          const int nchunks = grp.x, ntaps = grp.y;
          const uint32_t q0 = static_cast<uint32_t>(grp.w);
          const bool unrolled = g == 0 && g0_unrolled;
          for (int c = 0; c < nchunks; ++c) {
            mbar_wait_t(&a_full[as], aph, timed, w_afull);
            tc_fence_after();
            if (tile == 0 && g == 0 && c == 0 && timed) p.dbg[3] = clock64();
            const uint32_t a_win_lo = a_base_lo + as * a_slot_lo;
            if (unrolled) {
#pragma unroll
              for (int t = 0; t < kUnroll; ++t) {
                const uint32_t b_lo = b_acquire(q0 + t * nchunks + c);
                issue_step(a_win_lo + relu_[t], b_lo);
                b_release();
              }
            } else {
              const uint32_t* rel = s_rel + grp.z;
              for (int t = 0; t < ntaps; ++t) {
                const uint32_t b_lo = b_acquire(q0 + t * nchunks + c);
                issue_step(a_win_lo + rel[t], b_lo);
                b_release();
              }
            }
            commit(&a_empty[as]);            // window slot is free once all its taps retire
            if (++as == a_slots) { as = 0; aph ^= 1u; }
          }
        }
        commit(&acc_full[acc]);
        if (timed) {
          if (tile == 0) p.dbg[4] = clock64();
          if (tile + n_walkers >= total_tiles) p.dbg[9] = clock64();
        }
        if (++acc == acc_stages) { acc = 0; accph ^= 1u; }
      }
      if (timed) { p.dbg[18] = w_accempty; p.dbg[19] = w_afull; p.dbg[20] = w_bfull; }
    }
  } else if constexpr (EPI == 4) {
    // ===================== epilogue warps, fused ReLU + 3x3/2 max-pool (the stem) =====================
    // The tile is 3 consecutive conv rows (2i'-1, 2i', 2i'+1; 342 of the 384 accumulator rows) of one
    // image: every warp converts its TMEM block to bf16 (+bias, ReLU) into a swizzled
    // shared-memory conv tile, the 8 epilogue warps synchronise on a named barrier, then pool the
    // tile into pooled row i' (57 entries incl. the zero pad column) and write it -- the un-pooled
    // 112x112x64 map (1.6 MB per image) never goes to HBM.  Reference: models/cnn_backbone.py:349-354.
    static_assert(EPI != 4 || (BN == 64 && MT == 3), "pool epilogue is specialised for the stem");
    const int ew = warp - 2;
    const int quad = warp & 3, half = ew >> 2;
    const int tid = threadIdx.x - 64;                  // 0..255 within the epilogue warps
    uint8_t* ct = smem_stage;                          // conv tile: 384 rows x 128 B (64 bf16), 16-byte chunks XOR-swizzled by row
    const float* const bias = p.bias;
    const int acc_stages = p.acc_stages;
    const int cP = p.pool_P, Wo = p.pool_Wo, Ho = p.pool_Ho, Po = p.pool_Po, rpio = p.pool_rpio, tpi = p.tiles_per_img;
    uint4* const out = reinterpret_cast<uint4*>(p.out);
    const bool has_bias = bias != nullptr;             // the VQA stem folds its bias into K (ingest writes a 1 column)
    pdl_wait();                                        // the output buffer may still be read by a predecessor
    int acc = 0;
    uint32_t accph = 0;
    const bool timed = p.dbg != nullptr && blockIdx.x == 0 && warp == 2;
    long long w_accfull = 0;
    for (int tile = walker; tile < total_tiles; tile += n_walkers) {
      const int mt_idx = cta_mtile(tile);                      // this CTA's (image, pooled row) tile
      const bool real = mt_idx < p.m_tiles_cta;                // pair mode: the last pair may carry a phantom tile
      const int img = mt_idx / tpi, ip = mt_idx - img * tpi;   // image, pooled row
      mbar_wait_t(&acc_full[acc], accph, timed, w_accfull);
      tc_fence_after();
      if (warp == 2 && tile == walker) VQA_DBG(5);
      // No pad masking here: the pooling pass below only reads in-image conv positions.
      uint32_t v[MT][32];
      __syncwarp();
#pragma unroll
      for (int sub = 0; sub < MT; ++sub)
        tmem_ld32(tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + acc * (BN * MT) + sub * BN + half * 32, v[sub]);
      tmem_ld_wait();
      if (has_bias) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const float4 bq = __ldg(reinterpret_cast<const float4*>(bias + half * 32) + k);
#pragma unroll
          for (int sub = 0; sub < MT; ++sub) {
            v[sub][4 * k] = __float_as_uint(__uint_as_float(v[sub][4 * k]) + bq.x);
            v[sub][4 * k + 1] = __float_as_uint(__uint_as_float(v[sub][4 * k + 1]) + bq.y);
            v[sub][4 * k + 2] = __float_as_uint(__uint_as_float(v[sub][4 * k + 2]) + bq.z);
            v[sub][4 * k + 3] = __float_as_uint(__uint_as_float(v[sub][4 * k + 3]) + bq.w);
          }
        }
      }
#pragma unroll
      for (int sub = 0; sub < MT; ++sub) {
        const int rl = sub * 128 + quad * 32 + lane;     // row within the conv tile
        uint8_t* dst = ct + rl * 128;
#pragma unroll
        for (int c4 = 0; c4 < 4; ++c4) {
          uint32_t w[4];
#pragma unroll
          for (int k = 0; k < 4; ++k)
            w[k] = pack_relu_bf16x2(__uint_as_float(v[sub][8 * c4 + 2 * k]), __uint_as_float(v[sub][8 * c4 + 2 * k + 1]));
          *reinterpret_cast<uint4*>(dst + (((half * 4 + c4) ^ (rl & 7)) << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {                                     // TMEM stage drained: the next tile's MMAs may start
        if (PAIR) mbar_arrive_leader(&acc_empty[acc]); else mbar_arrive(&acc_empty[acc]);
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");       // conv tile complete (epilogue warps only)
      // ---- pooling pass: item = (pooled column j', channel octet cg)
      const size_t orow = static_cast<size_t>(img) * rpio + static_cast<size_t>(ip) * Po;
      for (int item = tid; item < (real ? Po * 8 : 0); item += 256) {
        const int jp = item >> 3, cg = item & 7;
        uint4 o = make_uint4(0u, 0u, 0u, 0u);
        if (jp < Wo) {
          __nv_bfloat162 m[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) m[k] = __float2bfloat162_rn(0.f);   // post-ReLU values are >= 0
#pragma unroll
          for (int r = 0; r < 3; ++r) {
            if (r == 0 && ip == 0) continue;                 // conv row -1 is padding (row 2i'+1 <= H-1 always holds)
#pragma unroll
            for (int dc = -1; dc <= 1; ++dc) {
              const int c = 2 * jp + dc;
              if (c < 0) continue;                           // column -1 is padding (c <= W-1 always holds)
              const int rl = r * cP + c;
              const uint4 q = *reinterpret_cast<const uint4*>(ct + rl * 128 + ((cg ^ (rl & 7)) << 4));
              const __nv_bfloat162* qv = reinterpret_cast<const __nv_bfloat162*>(&q);
#pragma unroll
              for (int k = 0; k < 4; ++k) m[k] = __hmax2(m[k], qv[k]);
            }
          }
          o = *reinterpret_cast<uint4*>(m);
        }
        out[(orow + jp) * 8 + cg] = o;
        if (ip == Ho - 1) out[(orow + Po + jp) * 8 + cg] = make_uint4(0u, 0u, 0u, 0u);   // the image's zero pad row
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");       // pooling done: the conv tile may be overwritten
      if (warp == 2 && tile == walker) VQA_DBG(6);
      if (warp == 2 && tile + n_walkers >= total_tiles) VQA_DBG(7);
      if (++acc == acc_stages) { acc = 0; accph ^= 1u; }
    }
    if (timed && lane == 0) p.dbg[21] = w_accfull;
  } else if constexpr (SF > 1) {
    // ===================== epilogue warps, shift-fused tiles (MT = 1, BN = 64, bf16 output) =====================
    // x[r] = sum_j acc_j[r + j*step] costs two warp shuffles and three adds per output on top of the usual bias /
    // residual / pack work: ~850 warp instructions per 128x64 tile and quadrant, against ~1150-1430 cycles of MMAs.
    // Measured with 8 epilogue warps (two per scheduler): 0.29 instructions per clock and scheduler, the epilogue and
    // not the tensor pipe sets the pace.  Hence 16 epilogue warps for these kernels, four per scheduler:
    //   warp = (group g, column half, TMEM lane quadrant); group g drains accumulator stage g, i.e. every other tile,
    //   so the two groups run one tile apart and their phases (TMEM loads, shuffles, staging, TMA) interleave;
    //   a warp owns 32 accumulator rows x 32 output channels, handled as two 16-channel passes to stay within the
    //   112 registers that 576 threads leave per thread.
    // Rows r + j*step >= 32 live in the next quadrant's slab: every warp publishes its first rows in shared memory,
    // and lanes < j*step (whose own rows nobody in this warp needs) pick up the next slab's rows, so ONE rotate-
    // shuffle per value serves all 32 lanes.  (tcgen05.shift was measured for this too: it shifts 8 columns by one
    // row inside each 32-lane quadrant in ~48 cycles of the tensor pipe -- 24 of them per tile cost as much as the
    // tile's MMAs; tools/ubench_shift.cu.)
    static_assert(BN == 64, "shift-fused epilogue: 64 output channels");
    constexpr bool kRes = (EPI & 1) != 0;
    constexpr int kSlotBytes = 32 * 64;       // 32 rows x 32 bf16 channels, SWIZZLE_64B
    const int ew = warp - 2;                  // 0..15
    const int quad = warp & 3;                // TMEM lane quadrant this warp may read
    const int grp = ew >> 3;                  // tile parity / accumulator stage this warp serves
    const int half = (ew >> 2) & 1;           // which 32 of the 64 output channels
    uint8_t* const out_slot = smem_stage + ew * ((kRes ? 2 : 1) * kSlotBytes);
    uint8_t* const res_slot = out_slot + kSlotBytes;
    uint64_t* const my_res_bar = &res_bar[ew];
    const uint32_t swz = (lane >> 1) & 3;     // SWIZZLE_64B: 16-byte unit u of row `lane` lives at ((u ^ swz) << 4)
    uint8_t* const out_row = out_slot + lane * 64;
    const uint8_t* const res_row = res_slot + lane * 64;
    const bool relu = p.relu != 0, mask_en = p.mask_en != 0, out_f16 = p.out_f16 != 0;
    const int step = p.sf_step;
    const bool has_bias = p.bias != nullptr;
    const int bar_id = 2 + (ew >> 2);         // named barrier of the four quadrant warps of this (group, half)
    for (int i = threadIdx.x - 64; i < BN; i += 32 * kSfEpiWarps) s_bias[i] = (has_bias && i < p.N) ? __ldg(p.bias + i) : 0.f;
    asm volatile("bar.sync 1, 512;" ::: "memory");
    pdl_wait();   // residual loads / output stores below touch buffers of the preceding kernels

    uint32_t accph = 0, resph = 0;
    int xpar = 0;
    const bool timed = p.dbg != nullptr && blockIdx.x == 0 && warp == 2;
    long long w_accfull = 0;
    long long ph_ld = 0, ph_xch = 0, ph_comb = 0, ph_fin = 0, ph_st = 0, ph_t = 0;   // epilogue phase cycles (dbg only)
#define VQA_PHASE(accu) do { if (timed) { const long long now__ = clock64(); accu += now__ - ph_t; ph_t = now__; } } while (0)
    const int tstep = 2 * n_walkers;          // this group's next tile
    const int first = walker + grp * n_walkers;
    auto issue_res = [&](int row0) {          // lane 0 only: 32 rows x 32 channels of the residual
      mbar_expect_tx(my_res_bar, kSlotBytes);
      tma_load_2d(res_slot, &mapRes, my_res_bar, 32 * half, row0);
    };
    if (kRes && lane == 0 && first < total_tiles) issue_res(tile_m0(p, cta_mtile(first), 1) + quad * 32);

    for (int tile = first; tile < total_tiles; tile += tstep) {
      const int row0 = tile_m0(p, cta_mtile(tile), 1) + quad * 32;
      const bool pix = !mask_en || grid_pixel(p, row0 + lane);
      const int ntile = tile + tstep;
      const int n_row0 = tile_m0(p, cta_mtile(ntile), 1) + quad * 32;
      mbar_wait_t(&acc_full[grp], accph, timed, w_accfull);
      accph ^= 1u;
      tc_fence_after();
      if (warp == 2 && tile == walker) VQA_DBG(5);
      if (timed) ph_t = clock64();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + grp * kAcc + 32 * half;
#pragma unroll 1
      for (int c = 0; c < 2; ++c) {           // 16-channel passes
        uint32_t v[SF][16];
        __syncwarp();                         // tcgen05.ld is .sync.aligned
#pragma unroll
        for (int j = 0; j < SF; ++j) tmem_ld16(taddr + j * BN + 16 * c, v[j]);
        if (kRes && c == 0) { mbar_wait(my_res_bar, resph); resph ^= 1u; }   // this tile's residual box has landed
        tmem_ld_wait();
        if (c == 1) {                         // every TMEM read of this warp is complete: release the accumulator stage
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if (PAIR) mbar_arrive_leader(&acc_empty[grp]); else mbar_arrive(&acc_empty[grp]);
          }
        }
        VQA_PHASE(ph_ld);
        // publish the first rows of blocks j >= 1 for the warp that owns the 32 rows before them
        float* const xmine = s_xchg + (((xpar * 4 + (ew >> 2)) * 4 + quad) * kXchgRows) * 16;
#pragma unroll
        for (int j = 1; j < SF; ++j) {
          if (lane < j * step) {
            float4* dst = reinterpret_cast<float4*>(xmine + (step * (j * (j - 1) / 2) + lane) * 16);
#pragma unroll
            for (int u = 0; u < 4; ++u)
              dst[u] = make_float4(__uint_as_float(v[j][4 * u]), __uint_as_float(v[j][4 * u + 1]),
                                   __uint_as_float(v[j][4 * u + 2]), __uint_as_float(v[j][4 * u + 3]));
          }
        }
        // split barrier: every thread arrives twice (here, after publishing, and in the bar.sync below), so the barrier
        // expects 2 x 128 arrivals and the work on block 0 overlaps the other warps' publishing
        asm volatile("bar.arrive %0, 256;" ::"r"(bar_id) : "memory");
        float x[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) x[k] = __uint_as_float(v[0][k]);
        if (has_bias) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float4 bq = *reinterpret_cast<const float4*>(s_bias + 32 * half + 16 * c + 4 * k);   // broadcast
            x[4 * k] += bq.x; x[4 * k + 1] += bq.y; x[4 * k + 2] += bq.z; x[4 * k + 3] += bq.w;
          }
        }
        if constexpr (kRes) {
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const uint4 q = *reinterpret_cast<const uint4*>(res_row + (((2 * c + u) ^ swz) << 4));
            const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              x[8 * u + 2 * k] += __uint_as_float(w[k] << 16);
              x[8 * u + 2 * k + 1] += __uint_as_float(w[k] & 0xFFFF0000u);
            }
          }
          if (c == 1) {
            __syncwarp();                     // every lane has consumed the residual slot: prefetch the next tile's box
            if (lane == 0 && ntile < total_tiles) issue_res(n_row0);
          }
        }
        VQA_PHASE(ph_fin);
        asm volatile("bar.sync %0, 256;" ::"r"(bar_id) : "memory");   // every quadrant warp has published
        VQA_PHASE(ph_xch);
        const float* const xnext = xmine + kXchgRows * 16;           // quadrant + 1; nothing for quadrant 3
#pragma unroll
        for (int j = 1; j < SF; ++j) {
          const int sh = j * step;
          if (lane < sh && quad < 3) {
            const float4* src = reinterpret_cast<const float4*>(xnext + (step * (j * (j - 1) / 2) + lane) * 16);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const float4 q = src[u];
              v[j][4 * u] = __float_as_uint(q.x); v[j][4 * u + 1] = __float_as_uint(q.y);
              v[j][4 * u + 2] = __float_as_uint(q.z); v[j][4 * u + 3] = __float_as_uint(q.w);
            }
          }
          const int from = (lane + sh) & 31;
#pragma unroll
          for (int k = 0; k < 16; ++k) x[k] += __shfl_sync(0xffffffffu, __uint_as_float(v[j][k]), from);
        }
        xpar ^= 1;
        VQA_PHASE(ph_comb);
        uint32_t w[8];
        if (out_f16) {
#pragma unroll
          for (int k = 0; k < 8; ++k) w[k] = relu ? pack_relu_f16x2(x[2 * k], x[2 * k + 1]) : pack_f16x2(x[2 * k], x[2 * k + 1]);
        } else {
#pragma unroll
          for (int k = 0; k < 8; ++k) w[k] = relu ? pack_relu_bf16x2(x[2 * k], x[2 * k + 1]) : pack_bf16x2(x[2 * k], x[2 * k + 1]);
        }
        if (!pix) {                           // keep the grid's shared zero padding intact
#pragma unroll
          for (int k = 0; k < 8; ++k) w[k] = 0u;
        }
        VQA_PHASE(ph_fin);
        if (c == 0) {
          if (lane == 0) bulk_wait_read0();   // the previous tile's TMA store has drained the out slot
          __syncwarp();
          VQA_PHASE(ph_st);
        }
#pragma unroll
        for (int u = 0; u < 2; ++u)
          *reinterpret_cast<uint4*>(out_row + (((2 * c + u) ^ swz) << 4)) = make_uint4(w[4 * u], w[4 * u + 1], w[4 * u + 2], w[4 * u + 3]);
      }
      fence_proxy_async();                    // staging writes -> visible to the TMA engine
      __syncwarp();
      if (lane == 0) {
        tma_store_2d(quad == 3 ? &mapOutLast : &mapOut, out_slot, 32 * half, row0);
        bulk_commit();
      }
      VQA_PHASE(ph_fin);
      if (warp == 2 && tile == walker) { VQA_DBG(13); VQA_DBG(6); }
      if (warp == 2 && tile + tstep >= total_tiles) VQA_DBG(7);
    }
    if (lane == 0) bulk_wait_all();           // outstanding TMA stores complete before the CTA exits
    if (timed && lane == 0) {
      p.dbg[21] = w_accfull;
      p.dbg[10] = ph_ld; p.dbg[11] = ph_xch; p.dbg[12] = ph_comb; p.dbg[14] = ph_fin; p.dbg[15] = ph_st;
    }
#undef VQA_PHASE
  } else {
    // ===================== epilogue warps =====================
    constexpr bool kOutBf16 = EPI < 2;
    constexpr bool kRes = (EPI & 1) != 0;
    constexpr bool kTopK = EPI == 6;    // fp32 output + fused softmax / top-k of the rows (MT = 1)
    static_assert(!kTopK || MT == 1, "the top-k epilogue is instantiated for MT = 1");
    constexpr int kCols = BN / 2;       // columns per epilogue warp (two warps share a lane quadrant)
    constexpr int kChunks = kCols / 32; // 32-column chunks per warp per sub-tile (1, 2 or 4)
    constexpr int kRowB = kOutBf16 ? 64 : 128;          // bytes of one chunk row in the staging slot
    constexpr int kUnits = kRowB / 16;                  // 16-byte units per row (4 / 8)
    constexpr int kSlotBytes = 32 * kRowB;
    const int ew = warp - 2;
    const int quad = warp & 3;          // TMEM lane quadrant this warp may read
    const int half = ew >> 2;           // which half of the tile's columns
    uint8_t* const out_slot = smem_stage + ew * ((kRes ? 2 : 1) * kSlotBytes);
    uint8_t* const res_slot = out_slot + kSlotBytes;
    uint64_t* const my_res_bar = &res_bar[ew];
    // this lane's row inside a slot: 16-byte unit u lives at row_off + ((u ^ swz) << 4)
    const uint32_t swz = kOutBf16 ? ((lane >> 1) & 3) : (lane & 7);
    uint8_t* const out_row = out_slot + lane * kRowB;
    const uint8_t* const res_row = res_slot + lane * kRowB;
    // loop-invariant parameters in registers (the asm volatile barriers would otherwise force reloads)
    const int N = p.N;
    const bool relu = p.relu != 0, rnd = p.round_tf32 != 0, mask_en = p.mask_en != 0, out_f16 = p.out_f16 != 0;
    const int m_tiles = p.m_tiles, acc_stages = p.acc_stages;
    const bool has_bias = p.bias != nullptr;
    float* const sums = p.sums;
    const int ld_sums = p.ld_sums;
    {   // bias of all N tiles -> shared memory (zero beyond N), read back as warp-wide broadcasts
      const int nb = min(p.n_tiles * BN, kBiasTable);
      for (int i = threadIdx.x - 64; i < nb; i += 32 * kEpiWarps) s_bias[i] = (has_bias && i < N) ? __ldg(p.bias + i) : 0.f;
      asm volatile("bar.sync 1, 256;" ::: "memory");
    }
    pdl_wait();   // residual loads / output stores below touch buffers of the preceding kernels

    int acc = 0;
    uint32_t accph = 0, resph = 0;
    const bool timed = p.dbg != nullptr && blockIdx.x == 0 && warp == 2;
    long long w_accfull = 0;
    long long ph_ld = 0, ph_fin = 0, ph_st = 0, ph_t = 0;   // epilogue phase cycles (dbg only)
#define VQA_PHASE(accu) do { if (timed) { const long long now__ = clock64(); accu += now__ - ph_t; ph_t = now__; } } while (0)
    const int tstep = n_walkers;

    auto issue_res = [&](int row0, int col0) {          // lane 0 only
      mbar_expect_tx(my_res_bar, kSlotBytes);
      tma_load_2d(res_slot, &mapRes, my_res_bar, col0, row0);
    };
    if (kRes && lane == 0 && walker < total_tiles) {
      issue_res(tile_m0(p, cta_mtile(walker), MT) + quad * 32, tile_nt(walker) * BN + half * kCols);
    }

    for (int tile = walker; tile < total_tiles; tile += tstep) {
      const int m0 = tile_m0(p, cta_mtile(tile), MT);
      const int n0 = tile_nt(tile) * BN;
      const int colw = n0 + half * kCols;               // first column this warp owns
      // ---- work that does not need the accumulator: done while the MMAs are still running
      bool pix[MT];
#pragma unroll
      for (int sub = 0; sub < MT; ++sub) {
        pix[sub] = true;
        if (mask_en) pix[sub] = grid_pixel(p, m0 + sub * 128 + quad * 32 + lane);
      }
      const int ntile = tile + tstep;                   // the residual of its first chunk is prefetched at the end
      const bool has_ntile = ntile < total_tiles;
      const int n_row0 = tile_m0(p, cta_mtile(ntile), MT) + quad * 32;
      const int n_col0 = tile_nt(ntile) * BN + half * kCols;

      // fused softmax / top-k (EPI 6): this thread's row over the columns this warp drains
      float tk_m = -INFINITY, tk_s = 0.f;
      bool tk_nan = false;
      float tk_v[kTopKMax];
      int tk_i[kTopKMax];
#pragma unroll
      for (int j = 0; j < kTopKMax; ++j) { tk_v[j] = -INFINITY; tk_i[j] = 0x7fffffff; }

      mbar_wait_t(&acc_full[acc], accph, timed, w_accfull);
      tc_fence_after();
      if (warp == 2 && tile == walker) VQA_DBG(5);
      if (timed) ph_t = clock64();
#pragma unroll
      for (int sub = 0; sub < MT; ++sub) {
        const int row0 = m0 + sub * 128 + quad * 32;
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + acc * (kAcc * MT) + sub * kAcc +
                               half * kCols;
#pragma unroll
        for (int c = 0; c < kChunks; ++c) {
          const int col0 = colw + 32 * c;               // first column of this 32-wide chunk (warp-uniform)
          if (!kRes && col0 >= N) continue;             // chunk entirely beyond N (the residual chain never skips)
          const bool tabled = p.n_tiles * BN <= kBiasTable;   // else (N > 2048): broadcast loads from global
          const float* bsrc = s_bias + (tabled ? col0 : 0);
          float x[32];
          uint32_t v[32];
          __syncwarp();                                 // tcgen05.ld is .sync.aligned
          tmem_ld32(taddr + 32 * c, v);
          if (kRes) mbar_wait(my_res_bar, resph);       // this chunk's residual box has landed
          tmem_ld_wait();
          VQA_PHASE(ph_ld);
#pragma unroll
          for (int k = 0; k < 32; ++k) x[k] = __uint_as_float(v[k]);
          if (has_bias && !tabled) {
#pragma unroll
            for (int k = 0; k < 32; ++k) x[k] += (col0 + k < N) ? __ldg(p.bias + col0 + k) : 0.f;
          } else if (has_bias) {
#pragma unroll
            for (int k = 0; k < 8; ++k) {
              const float4 bq = *reinterpret_cast<const float4*>(bsrc + 4 * k);   // same address in every lane: broadcast
              x[4 * k] += bq.x; x[4 * k + 1] += bq.y; x[4 * k + 2] += bq.z; x[4 * k + 3] += bq.w;
            }
          }
          if constexpr (kRes) {
            resph ^= 1u;
#pragma unroll
            for (int u = 0; u < kUnits; ++u) {
              const uint4 q = *reinterpret_cast<const uint4*>(res_row + ((u ^ swz) << 4));
              if constexpr (kOutBf16) {
                const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  x[8 * u + 2 * k] += __uint_as_float(w[k] << 16);
                  x[8 * u + 2 * k + 1] += __uint_as_float(w[k] & 0xFFFF0000u);
                }
              } else {
                x[4 * u] += __uint_as_float(q.x); x[4 * u + 1] += __uint_as_float(q.y);
                x[4 * u + 2] += __uint_as_float(q.z); x[4 * u + 3] += __uint_as_float(q.w);
              }
            }
            __syncwarp();                               // every lane has consumed the residual slot
            if (lane == 0) {                            // prefetch the next chunk's residual box
              const bool last = (sub == MT - 1) && (c == kChunks - 1);
              if (!last) issue_res(m0 + ((c + 1 < kChunks) ? sub : sub + 1) * 128 + quad * 32,
                                   colw + 32 * ((c + 1 < kChunks) ? c + 1 : 0));
              else if (has_ntile) issue_res(n_row0, n_col0);
            }
          }
          VQA_PHASE(ph_fin);
          if (lane == 0) bulk_wait_read0();             // the previous chunk's TMA store has drained the out slot
          __syncwarp();
          VQA_PHASE(ph_st);
          if constexpr (kOutBf16) {
            uint32_t w[16];
            if (out_f16) {
              if (relu) {
#pragma unroll
                for (int k = 0; k < 16; ++k) w[k] = pack_relu_f16x2(x[2 * k], x[2 * k + 1]);
              } else {
#pragma unroll
                for (int k = 0; k < 16; ++k) w[k] = pack_f16x2(x[2 * k], x[2 * k + 1]);
              }
            } else if (relu) {
#pragma unroll
              for (int k = 0; k < 16; ++k) w[k] = pack_relu_bf16x2(x[2 * k], x[2 * k + 1]);
            } else {
#pragma unroll
              for (int k = 0; k < 16; ++k) w[k] = pack_bf16x2(x[2 * k], x[2 * k + 1]);
            }
            if (!pix[sub]) {                            // keep the grid's shared zero padding intact
#pragma unroll
              for (int k = 0; k < 16; ++k) w[k] = 0u;
            }
#pragma unroll
            for (int u = 0; u < kUnits; ++u)
              *reinterpret_cast<uint4*>(out_row + ((u ^ swz) << 4)) = make_uint4(w[4 * u], w[4 * u + 1], w[4 * u + 2], w[4 * u + 3]);
            if (sums != nullptr) {                      // SE squeeze partial sums of this 32-row slab (warp-uniform branch)
              const bool live = pix[sub] && row0 + lane < p.M;     // rows past M exist only in the accumulator
#pragma unroll
              for (int k = 0; k < 32; ++k) x[k] = live ? (relu ? relu_f32(x[k]) : x[k]) : 0.f;
              const float tot = warp_colsum32(x, lane);
              if (row0 < p.M && col0 + lane < N) sums[static_cast<size_t>(row0 >> 5) * ld_sums + col0 + lane] = tot;
            }
          } else {
            if (relu) {
#pragma unroll
              for (int k = 0; k < 32; ++k) x[k] = relu_f32(x[k]);
            }
            if (!pix[sub]) {
#pragma unroll
              for (int k = 0; k < 32; ++k) x[k] = 0.f;
            }
            if (TF32 && rnd) {
#pragma unroll
              for (int k = 0; k < 32; ++k) x[k] = round_tf32_rna(x[k]);
            }
            if constexpr (kTopK) {
              // online softmax statistics (max ignores NaN like fmaxf, the sum turns NaN like the reference's) and the
              // k best of the stored values in rank_before's order (NaN above everything, torch.topk's order)
              float cm = -INFINITY;
#pragma unroll
              for (int k = 0; k < 32; ++k) {
                if (col0 + k < N) { if (x[k] != x[k]) tk_nan = true; else cm = fmaxf(cm, x[k]); }
              }
              const float m_new = fmaxf(tk_m, cm);
              if (m_new > -INFINITY) {
                float add = 0.f;
#pragma unroll
                for (int k = 0; k < 32; ++k) {
                  if (col0 + k < N && x[k] == x[k]) add += expf(x[k] - m_new);
                }
                tk_s = tk_s * expf(tk_m - m_new) + add;
                tk_m = m_new;
              }
#pragma unroll
              for (int k = 0; k < 32; ++k) {
                if (col0 + k < N) topk_insert(tk_v, tk_i, x[k], col0 + k);
              }
            }
#pragma unroll
            for (int u = 0; u < kUnits; ++u)
              *reinterpret_cast<float4*>(out_row + ((u ^ swz) << 4)) = make_float4(x[4 * u], x[4 * u + 1], x[4 * u + 2], x[4 * u + 3]);
          }
          fence_proxy_async();                          // staging writes -> visible to the TMA engine
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&mapOut, out_slot, col0, row0);
            bulk_commit();
          }
          VQA_PHASE(ph_fin);
        }
      }
      if (warp == 2 && tile == walker) VQA_DBG(13);
      // all TMEM reads of this warp are complete (wait::ld above): release the accumulator stage
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (PAIR) mbar_arrive_leader(&acc_empty[acc]); else mbar_arrive(&acc_empty[acc]);
      }
      if constexpr (kTopK) {
        // ---- publish this thread's partial (one 80-byte record: max, exp-sum, pad, pad, 8 keys, 8 indices); the CTA that
        // completes the M tile's last N tile merges the row: thread (row, half) folds the records of every other slot
        // (vector loads, the next record in flight while the current one is inserted), the two halves meet in shared memory
        const int nparts = 2 * p.n_tiles, mt_idx = tile_mt(tile);
        const int row = m0 + quad * 32 + lane;
        if (row < p.M) {
          float4* rec = reinterpret_cast<float4*>(p.topk_part + (static_cast<size_t>(row) * nparts + tile_nt(tile) * 2 + half) * kTopKRec);
          rec[0] = make_float4(tk_m, tk_nan ? __int_as_float(0x7fc00000) : tk_s, 0.f, 0.f);
          rec[1] = make_float4(tk_v[0], tk_v[1], tk_v[2], tk_v[3]);
          rec[2] = make_float4(tk_v[4], tk_v[5], tk_v[6], tk_v[7]);
          rec[3] = make_float4(__int_as_float(tk_i[0]), __int_as_float(tk_i[1]), __int_as_float(tk_i[2]), __int_as_float(tk_i[3]));
          rec[4] = make_float4(__int_as_float(tk_i[4]), __int_as_float(tk_i[5]), __int_as_float(tk_i[6]), __int_as_float(tk_i[7]));
        }
        __threadfence();
        asm volatile("bar.sync 1, 256;" ::: "memory");
        volatile uint32_t* last_flag = tmem_slot + 1;
        if (threadIdx.x == 64) *last_flag = (atomicAdd(p.topk_cnt + mt_idx, 1) == p.n_tiles - 1) ? 1u : 0u;
        asm volatile("bar.sync 1, 256;" ::: "memory");
        if (*last_flag != 0u) {
          __threadfence();
          float gm = -INFINITY, gs = 0.f;
          float bv[kTopKMax];
          int bi[kTopKMax];
#pragma unroll
          for (int j = 0; j < kTopKMax; ++j) { bv[j] = -INFINITY; bi[j] = 0x7fffffff; }
          auto fold = [&](const float4 (&r)[5]) {            // online merge of one record into (gm, gs, bv, bi)
            const float pm = r[0].x, ps = r[0].y;
            const float nm = fmaxf(gm, pm);
            if (ps != ps) gs = ps;                            // a NaN anywhere in the row: the softmax denominator is NaN
            else if (nm > -INFINITY && gs == gs) gs = gs * expf(gm - nm) + ps * expf(pm - nm);
            gm = nm;
            const float kv[8] = {r[1].x, r[1].y, r[1].z, r[1].w, r[2].x, r[2].y, r[2].z, r[2].w};
            const float ki[8] = {r[3].x, r[3].y, r[3].z, r[3].w, r[4].x, r[4].y, r[4].z, r[4].w};
#pragma unroll
            for (int j = 0; j < kTopKMax; ++j) topk_insert(bv, bi, kv[j], __float_as_int(ki[j]));
          };
          if (row < p.M) {
            const float4* rec = reinterpret_cast<const float4*>(p.topk_part + static_cast<size_t>(row) * nparts * kTopKRec);
            float4 cur[5], nxt[5];
#pragma unroll
            for (int u = 0; u < 5; ++u) cur[u] = __ldcg(rec + half * 5 + u);
            for (int q = half; q < nparts; q += 2) {
              const bool more = q + 2 < nparts;
#pragma unroll
              for (int u = 0; u < 5; ++u) nxt[u] = more ? __ldcg(rec + (q + 2) * 5 + u) : make_float4(0.f, 0.f, 0.f, 0.f);
              fold(cur);
#pragma unroll
              for (int u = 0; u < 5; ++u) cur[u] = nxt[u];
            }
          }
          // the half-1 thread hands its merged record to the half-0 thread of the same row through its staging slot
          if (lane == 0) bulk_wait_read0();                   // this warp's last TMA store has drained the slot
          __syncwarp();
          float4* xrow = reinterpret_cast<float4*>(smem_stage + (ew | 4) * kSlotBytes + lane * kRowB);   // the half-1 warp's slot
          if (half == 1) {
            xrow[0] = make_float4(gm, gs, 0.f, 0.f);
            xrow[1] = make_float4(bv[0], bv[1], bv[2], bv[3]);
            xrow[2] = make_float4(bv[4], bv[5], bv[6], bv[7]);
            xrow[3] = make_float4(__int_as_float(bi[0]), __int_as_float(bi[1]), __int_as_float(bi[2]), __int_as_float(bi[3]));
            xrow[4] = make_float4(__int_as_float(bi[4]), __int_as_float(bi[5]), __int_as_float(bi[6]), __int_as_float(bi[7]));
          }
          asm volatile("bar.sync 1, 256;" ::: "memory");
          if (half == 0 && row < p.M) {
            const float4 r[5] = {xrow[0], xrow[1], xrow[2], xrow[3], xrow[4]};
            fold(r);
            const int kk = p.topk_k;
#pragma unroll
            for (int t = 0; t < kTopKMax; ++t) {
              if (t < kk) {
                int ii = bi[t];
                if (ii < 0 || ii >= N) ii = t < N ? t : N - 1;      // cannot happen with k <= N; never an out-of-row index
                p.topk_idx[static_cast<size_t>(row) * kk + t] = ii;
                p.topk_probs[static_cast<size_t>(row) * kk + t] = expf(bv[t] - gm) / gs;
              }
            }
          }
          if (threadIdx.x == 64) p.topk_cnt[mt_idx] = 0;          // ready for the next launch (CUDA-graph replay)
          asm volatile("bar.sync 1, 256;" ::: "memory");           // the staging slots are free again for the next tile
        }
      }
      if (warp == 2 && tile == walker) VQA_DBG(6);
      if (warp == 2 && tile + tstep >= total_tiles) VQA_DBG(7);
      if (++acc == acc_stages) { acc = 0; accph ^= 1u; }
    }
    if (lane == 0) bulk_wait_all();                     // outstanding TMA stores complete before the CTA exits
    if (timed && lane == 0) {
      p.dbg[21] = w_accfull;
      p.dbg[10] = ph_ld; p.dbg[11] = 0; p.dbg[12] = 0; p.dbg[14] = ph_fin; p.dbg[15] = ph_st;
    }
#undef VQA_PHASE
  }

  tc_fence_before();
  if (PAIR) cluster_sync(); else __syncthreads();       // pair: the leader's last commits land on the peer's barriers
  if (warp == 2) {
    if (PAIR) tmem_dealloc_pair(tmem_base, tmem_cols); else tmem_dealloc(tmem_base, tmem_cols);
  }
  if (warp == 0) VQA_DBG(8);
  if (p.dbg && blockIdx.x == 0 && threadIdx.x == 0) {
    unsigned long long ns;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(ns));
    p.dbg[23] = static_cast<long long>(ns);
  }
}

// ----------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* sym = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) != cudaSuccess ||
      qres != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(sym);
  return fn;
}

// 2-D K-major tensor map: dim0 = cols (contiguous), dim1 = rows with stride ld elements;
// box = {row_bytes, box_rows}, SWIZZLE_128B / SWIZZLE_32B to match row_bytes, out-of-range elements read as zero.
int encode_2d(CUtensorMap* map, bool tf32, uint64_t base, int rows, int cols, int ld, int box_rows, int row_bytes,
              const char* what) {
  EncodeTiledFn fn = get_encode_fn();
  VQA_REQUIRE(fn != nullptr, VQA_E_CUDA, "cuTensorMapEncodeTiled entry point not found");
  const int esz = tf32 ? 4 : 2;
  VQA_REQUIRE((base & 15) == 0, VQA_E_ALIGN, std::string(what) + ": tensor base must be 16-byte aligned");
  VQA_REQUIRE((static_cast<long long>(ld) * esz) % 16 == 0, VQA_E_ALIGN,
              std::string(what) + ": row stride must be a multiple of 16 bytes");
  VQA_REQUIRE(box_rows >= 1 && box_rows <= 256, VQA_E_INVALID, std::string(what) + ": box rows out of range");
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * esz};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(row_bytes / esz), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, tf32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2,
                  reinterpret_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    vqa_set_error(std::string(what) + ": cuTensorMapEncodeTiled failed with CUresult " + std::to_string(static_cast<int>(r)) +
                  " (rows=" + std::to_string(rows) + " cols=" + std::to_string(cols) + " ld=" + std::to_string(ld) +
                  " box_rows=" + std::to_string(box_rows) + ")");
    return VQA_E_CUDA;
  }
  return VQA_OK;
}

// Epilogue tensor map over the output (or residual) matrix: 32 x 32 element boxes, SWIZZLE_64B for bf16
// (64-byte box rows) / SWIZZLE_128B for fp32 (128-byte box rows), matching the staging slots of the kernel.
int encode_box32(CUtensorMap* map, bool f32, uint64_t base, int rows, int cols, int ld, const char* what, int box_rows = 32,
                 int box_cols = 32) {
  EncodeTiledFn fn = get_encode_fn();
  VQA_REQUIRE(fn != nullptr, VQA_E_CUDA, "cuTensorMapEncodeTiled entry point not found");
  const int esz = f32 ? 4 : 2;
  VQA_REQUIRE(base != 0 && (base & 15) == 0, VQA_E_ALIGN, std::string(what) + ": base must be 16-byte aligned");
  VQA_REQUIRE((static_cast<long long>(ld) * esz) % 16 == 0 && ld >= cols, VQA_E_ALIGN,
              std::string(what) + ": leading dimension must be >= N and a multiple of 16 bytes");
  // measured on B200: a TMA store clips the N edge in whole 16-byte granules, so a ragged last granule
  // would overwrite up to 3 elements of padding
  VQA_REQUIRE((static_cast<long long>(cols) * esz) % 16 == 0, VQA_E_ALIGN,
              std::string(what) + ": N must be a multiple of 16 bytes (4 fp32 / 8 bf16 columns)");
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * esz};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(box_cols), static_cast<cuuint32_t>(box_rows)};
  const bool sw128 = box_cols * esz == 128;     // 128-byte box rows: SWIZZLE_128B, 64-byte rows: SWIZZLE_64B
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2,
                  reinterpret_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  sw128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    vqa_set_error(std::string(what) + ": cuTensorMapEncodeTiled failed with CUresult " + std::to_string(static_cast<int>(r)));
    return VQA_E_CUDA;
  }
  return VQA_OK;
}

// UMMA instruction descriptor (cute::UMMA::InstrDescriptor bit layout): c_format f32 [4,6)=1,
// a/b format [7,10)/[10,13) (1 = bf16, 2 = tf32), K-major A and B, N>>3 at [17,23), M>>4 at [24,29).
uint32_t make_idesc(bool tf32, bool f16, int n, int m) {
  const uint32_t fmt = tf32 ? 2u : (f16 ? 0u : 1u);     // kind::f16: 0 = fp16, 1 = bf16; kind::tf32: 2
  return (1u << 4) | (fmt << 7) | (fmt << 10) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}

int num_sms(int device) {
  static int cached[64] = {0};
  if (device >= 0 && device < 64 && cached[device]) return cached[device];
  int n = 148;
  cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device);
  if (device >= 0 && device < 64) cached[device] = n;
  return n;
}

}  // namespace

// shared with stem_tcgen05.cu
int vqa_encode_2d(CUtensorMap* map, bool tf32, uint64_t base, int rows, int cols, int ld, int box_rows, int row_bytes,
                  const char* what) {
  return encode_2d(map, tf32, base, rows, cols, ld, box_rows, row_bytes, what);
}
int vqa_encode_box32f(CUtensorMap* map, uint64_t base, int rows, int cols, int ld, const char* what) {
  return encode_box32(map, true, base, rows, cols, ld, what);
}
int vqa_num_sms(int device) { return num_sms(device); }
uint32_t vqa_make_idesc(bool tf32, bool f16, int n, int m) { return make_idesc(tf32, f16, n, m); }

typedef void (*GemmKernelFn)(const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap,
                             const CUtensorMap, const CUtensorMap, const GemmParams);

// Instantiated (BN, MT, operand type, epilogue) combinations: bf16 kernels with epilogues 0/1/2
// (convolutions, image projector), tf32 kernels with MT = 1 and epilogues 2/3 (all nn.Linear layers).
static GemmKernelFn pick_kernel(int bn, int mt, bool tf32, int epi, int row_bytes, bool pair, int sf) {
#define VQA_K(BN_, MT_, TF_, EPI_, R32_, PAIR_) static_cast<GemmKernelFn>(&gemm_tap_kernel<BN_, MT_, TF_, EPI_, R32_, PAIR_>)
  if (sf > 1) {   // shift-fused 64-channel convolutions: N = sf * 64 MMAs, bf16 output with / without residual
    if (bn != 64 || mt != 1 || tf32 || row_bytes != 128 || epi > 1) return nullptr;
#define VQA_KSF(EPI_, PAIR_, SF_) static_cast<GemmKernelFn>(&gemm_tap_kernel<64, 1, false, EPI_, false, PAIR_, SF_>)
    if (sf == 3) return pair ? (epi ? VQA_KSF(1, true, 3) : VQA_KSF(0, true, 3)) : (epi ? VQA_KSF(1, false, 3) : VQA_KSF(0, false, 3));
    if (sf == 2) return pair ? (epi ? VQA_KSF(1, true, 2) : VQA_KSF(0, true, 2)) : (epi ? VQA_KSF(1, false, 2) : VQA_KSF(0, false, 2));
#undef VQA_KSF
    return nullptr;
  }
  if (row_bytes == 32) {   // the stem: 32-byte rows, bf16, N = 64, ReLU epilogue without residual
    if (pair) {
      if (bn == 64 && mt == 3 && !tf32 && epi == 4) return VQA_K(64, 3, false, 4, true, true);
      if (bn == 64 && mt == 2 && !tf32 && epi == 0) return VQA_K(64, 2, false, 0, true, true);
      return nullptr;
    }
    if (bn == 64 && mt == 1 && !tf32 && epi == 0) return VQA_K(64, 1, false, 0, true, false);
    if (bn == 64 && mt == 2 && !tf32 && epi == 0) return VQA_K(64, 2, false, 0, true, false);
    if (bn == 64 && mt == 2 && !tf32 && epi == 2) return VQA_K(64, 2, false, 2, true, false);
    if (bn == 64 && mt == 3 && !tf32 && epi == 4) return VQA_K(64, 3, false, 4, true, false);
    return nullptr;
  }
#define VQA_PICK(BN_, MT_, TF_, EPI_, PAIR_) \
  if (bn == BN_ && mt == MT_ && tf32 == TF_ && epi == EPI_ && pair == PAIR_) return VQA_K(BN_, MT_, TF_, EPI_, false, PAIR_);
#define VQA_PICK_BF16(BN_, MT_) VQA_PICK(BN_, MT_, false, 0, false) VQA_PICK(BN_, MT_, false, 1, false) \
  VQA_PICK(BN_, MT_, false, 2, false) VQA_PICK(BN_, MT_, false, 0, true) VQA_PICK(BN_, MT_, false, 1, true)
#define VQA_PICK_F16RES(BN_) VQA_PICK(BN_, 1, false, 3, false)   /* 16-bit operands, fp32 out + fp32 residual (fp16 tail) */
#define VQA_PICK_TF32(BN_) VQA_PICK(BN_, 1, true, 2, false) VQA_PICK(BN_, 1, true, 3, false)
  VQA_PICK(128, 1, false, 6, false)   /* 16-bit operands, fp32 out + fused softmax / top-k (answer head) */
  VQA_PICK_BF16(64, 1) VQA_PICK_BF16(64, 2) VQA_PICK_BF16(128, 1) VQA_PICK_BF16(128, 2)
  VQA_PICK_BF16(256, 1) VQA_PICK_BF16(256, 2)
  VQA_PICK_TF32(64) VQA_PICK_TF32(128) VQA_PICK_TF32(256)
  VQA_PICK_F16RES(64) VQA_PICK_F16RES(128) VQA_PICK_F16RES(256)
#undef VQA_PICK_F16RES
#undef VQA_PICK_TF32
#undef VQA_PICK_BF16
#undef VQA_PICK
#undef VQA_K
  return nullptr;
}

struct GemmLaunch {
  GemmKernelFn fn;
  int epi;
  CUtensorMap mapA0, mapA1, mapB, mapOut, mapRes, mapOutLast;
  bool out_external;    // the output is a caller tensor (logits): its map is encoded per run
  bool pair;            // CTA-pair (cta_group::2) launch: clusters of 2
  GemmParams prm;
  dim3 grid;
  int bn;
  int threads;          // CTA size: 10 warps, 18 for the shift-fused kernels
  size_t smem;
  uint64_t out_raw, res_raw, topk_idx_raw, topk_probs_raw;
};

int gemm_launch_bytes() { return static_cast<int>(sizeof(GemmLaunch)); }

int gemm_prepare(const VqaOp& op, void* storage, int device) {
  GemmLaunch* L = new (storage) GemmLaunch();
  GemmParams& p = L->prm;
  const int32_t* I = op.i;
  const bool tf32 = I[GEMM_I_dtype] == 1;
  const bool f16 = I[GEMM_I_dtype] == 2;                 // fp16 operands: same kernels as bf16, other format code
  const int bn = I[GEMM_I_BN];
  VQA_REQUIRE(bn == 64 || bn == 128 || bn == 256, VQA_E_INVALID, "gemm: BN must be 64, 128 or 256");
  p.M = I[GEMM_I_M];
  p.N = I[GEMM_I_N];
  p.MT = I[GEMM_I_MT];
  p.halo = I[GEMM_I_halo];
  VQA_REQUIRE(p.MT >= 1 && p.MT <= 3, VQA_E_INVALID, "gemm: MT must be 1, 2 or 3");
  const int sf = I[GEMM_I_sf] > 1 ? I[GEMM_I_sf] : 1;   // shift-fused form: sf column blocks of bn per MMA
  const int n_mma = sf * bn;
  p.sf_step = I[GEMM_I_sf_step] > 0 ? I[GEMM_I_sf_step] : 1;
  VQA_REQUIRE(p.MT * n_mma <= 512, VQA_E_INVALID, "gemm: accumulators exceed 512 TMEM columns");
  VQA_REQUIRE(sf == 1 || (sf <= 3 && p.MT == 1 && bn == 64 && I[GEMM_I_out_dtype] != 1 && p.N <= bn && I[GEMM_I_Npad] == n_mma &&
                          p.sf_step * (sf * (sf - 1) / 2) <= kXchgRows && (sf - 1) * p.sf_step < 32),
              VQA_E_INVALID, "gemm: shift-fused form needs MT = 1, N <= BN, Npad = sf * BN <= 256 and at most 4 exchanged rows");
  VQA_REQUIRE(p.M > 0 && p.N > 0 && I[GEMM_I_Npad] % bn == 0 && I[GEMM_I_Npad] >= p.N, VQA_E_INVALID,
              "gemm: bad M/N/Npad");
  p.ngroups = I[GEMM_I_ngroups];
  VQA_REQUIRE(p.ngroups >= 1 && p.ngroups <= VQA_MAX_GROUPS, VQA_E_INVALID, "gemm: bad group count");
  VQA_REQUIRE(I[GEMM_I_ntaps] >= 1 && I[GEMM_I_ntaps] <= VQA_MAX_TAPS, VQA_E_INVALID, "gemm: bad tap count");
  p.row_bytes = I[GEMM_I_row_bytes] > 0 ? I[GEMM_I_row_bytes] : 128;
  VQA_REQUIRE(p.row_bytes == 128 || (p.row_bytes == 32 && !tf32), VQA_E_INVALID, "gemm: row_bytes must be 128 (or 32 for bf16)");
  const int halo_hi = I[GEMM_I_halo_hi];
  VQA_REQUIRE(p.halo >= 0 && halo_hi >= 0, VQA_E_INVALID, "gemm: negative halo");
  p.chunk_elems = p.row_bytes / (tf32 ? 4 : 2);
  p.is_tf32 = tf32 ? 1 : 0;
  // UMMA shared-memory descriptor high word: SBO (8 rows) >> 4 at [32,46), version 1 at [46,48),
  // swizzle mode at [61,64): 2 = SWIZZLE_128B, 6 = SWIZZLE_32B
  p.desc_hi = static_cast<uint32_t>((8 * p.row_bytes) >> 4) | (1u << 14) | ((p.row_bytes == 128 ? 2u : 6u) << 29);
  const bool pair = I[GEMM_I_pair] != 0;
  L->pair = pair;
  // (tf32 pairs were measured too: no gain for the latency-bound M = 5120 Linears, so they are not instantiated)
  VQA_REQUIRE(!pair || (!tf32 && bn % 16 == 0), VQA_E_INVALID, "gemm: CTA pairs are instantiated for bf16 operands");
  p.idesc = make_idesc(tf32, f16, n_mma, pair ? 256 : 128);
  VQA_REQUIRE(I[GEMM_I_Ktot] % p.chunk_elems == 0, VQA_E_INVALID, "gemm: Ktot must be a multiple of the K chunk");
  p.k_chunks = I[GEMM_I_Ktot] / p.chunk_elems;
  bool lockstep = p.halo == 0 && halo_hi == 0;
  long long kcover = 0;
  bool uses_a1 = false;
  for (int g = 0; g < p.ngroups; ++g) {
    p.g_map[g] = I[GEMM_I_g_map0 + g];
    p.g_delta[g] = I[GEMM_I_g_delta0 + g];
    p.g_acol[g] = I[GEMM_I_g_acol0 + g];
    p.g_chunks[g] = I[GEMM_I_g_chunks0 + g];
    p.g_ntaps[g] = I[GEMM_I_g_ntaps0 + g];
    p.g_kbase[g] = I[GEMM_I_g_kbase0 + g];
    p.g_tap0[g] = I[GEMM_I_g_tap00 + g];
    VQA_REQUIRE(p.g_chunks[g] >= 1 && p.g_ntaps[g] >= 1 && p.g_tap0[g] + p.g_ntaps[g] <= VQA_MAX_TAPS,
                VQA_E_INVALID, "gemm: bad group");
    VQA_REQUIRE(p.g_kbase[g] % p.chunk_elems == 0, VQA_E_INVALID, "gemm: group K base must be chunk aligned");
    if (p.g_ntaps[g] != 1) lockstep = false;
    uses_a1 |= p.g_map[g] != 0;
    p.g_q0[g] = p.g_kbase[g] / p.chunk_elems;
    kcover += static_cast<long long>(p.g_ntaps[g]) * p.g_chunks[g] * p.chunk_elems;
  }
  VQA_REQUIRE(kcover == I[GEMM_I_Ktot], VQA_E_INVALID, "gemm: groups do not cover Ktot");
  p.win_per_tile = p.steps_per_tile = 0;
  for (int g = 0; g < p.ngroups; ++g) {
    p.win_per_tile += p.g_chunks[g];
    p.steps_per_tile += p.g_chunks[g] * p.g_ntaps[g];
  }
  for (int t = 0; t < VQA_MAX_TAPS; ++t) {
    p.tap_rel[t] = I[GEMM_I_tap_rel0 + t];
    VQA_REQUIRE(t >= I[GEMM_I_ntaps] || (p.tap_rel[t] >= 0 && p.tap_rel[t] <= p.halo + halo_hi), VQA_E_INVALID,
                "gemm: tap offset outside the window");
  }
  // window geometry
  const int win = 128 * p.MT + p.halo + halo_hi;
  p.nboxes = (win + 255) / 256;
  VQA_REQUIRE(p.nboxes <= 3, VQA_E_INVALID, "gemm: halo too large for a 3-box window");
  p.box_rows = ((win + p.nboxes - 1) / p.nboxes + 7) / 8 * 8;    // 8-row groups keep every box swizzle-aligned
  p.a_tx_bytes = p.nboxes * p.box_rows * p.row_bytes;
  p.a_slot_bytes = (p.a_tx_bytes + 1023) / 1024 * 1024;
  p.b_slot_bytes = (pair ? n_mma / 2 : n_mma) * p.row_bytes;    // pair: each CTA holds half of the weight tile's rows
  VQA_REQUIRE(p.b_slot_bytes % 1024 == 0, VQA_E_INVALID, "gemm: weight tile must be a multiple of 1024 bytes");
  p.m_tiles = (p.M + 128 * p.MT - 1) / (128 * p.MT);
  p.tiles_per_img = I[GEMM_I_tiles_per_img];
  p.tile_stride = I[GEMM_I_tile_stride];
  p.tile_row0 = I[GEMM_I_tile_row0];
  p.img_rows = I[GEMM_I_img_rows];
  const bool pool = I[GEMM_I_pool] != 0;
  if (p.tiles_per_img > 0) {
    VQA_REQUIRE(p.img_rows > 0 && p.tile_stride > 0 && I[GEMM_I_n_imgs] > 0, VQA_E_INVALID, "gemm: bad strided tiling");
    p.m_tiles = p.tiles_per_img * I[GEMM_I_n_imgs];
  }
  p.m_tiles_cta = p.m_tiles;
  if (pair) p.m_tiles = (p.m_tiles + 1) / 2;               // the kernel walks pairs of m tiles
  p.pool_P = I[GEMM_I_pool_P]; p.pool_W = I[GEMM_I_pool_W]; p.pool_Wo = I[GEMM_I_pool_Wo]; p.pool_Ho = I[GEMM_I_pool_Ho];
  p.pool_Po = I[GEMM_I_pool_Po]; p.pool_rpio = I[GEMM_I_pool_rpio];
  if (pool) {
    VQA_REQUIRE(p.MT == 3 && bn == 64 && p.row_bytes == 32 && p.tiles_per_img == p.pool_Ho && 3 * p.pool_P <= 384 &&
                    p.pool_Wo * 2 == p.pool_W && p.pool_Po >= p.pool_Wo + 1 && p.tile_stride == 2 * p.pool_P &&
                    p.tile_row0 == -p.pool_P, VQA_E_INVALID,
                "gemm: the fused max-pool epilogue needs 3 conv rows per tile (MT=3, BN=64, 32-byte rows)");
  }
  p.n_tiles = (p.N + bn - 1) / bn;        // only N tiles that contain real columns run
  p.acc_stages = (2 * p.MT * n_mma <= 512) ? 2 : 1;

  const bool has_res = op.p[GEMM_P_res] != 0;
  p.out_dtype = I[GEMM_I_out_dtype];
  p.res_dtype = I[GEMM_I_res_dtype];
  VQA_REQUIRE(!has_res || p.res_dtype == p.out_dtype, VQA_E_INVALID, "gemm: the residual must have the output's dtype");
  VQA_REQUIRE(p.out_dtype >= 0 && p.out_dtype <= 2, VQA_E_INVALID, "gemm: out_dtype must be 0 (bf16), 1 (fp32) or 2 (fp16)");
  p.out_f16 = p.out_dtype == 2 ? 1 : 0;
  L->epi = pool ? 4 : (p.out_dtype != 1 ? 0 : 2) + (has_res ? 1 : 0);
  {
    static const int pdl_late = std::getenv("VQA_PDL_LATE") ? std::atoi(std::getenv("VQA_PDL_LATE")) : 0;
    p.pdl_late = pdl_late;
  }
  p.topk_k = I[GEMM_I_topk];
  L->topk_idx_raw = op.p[GEMM_P_topk_idx];
  L->topk_probs_raw = op.p[GEMM_P_topk_probs];
  p.topk_part = reinterpret_cast<float*>(op.p[GEMM_P_topk_part]);
  p.topk_cnt = reinterpret_cast<int*>(op.p[GEMM_P_topk_cnt]);
  p.topk_idx = nullptr;
  p.topk_probs = nullptr;
  if (p.topk_k > 0) {
    VQA_REQUIRE(L->epi == 2 && !tf32 && bn == 128 && p.MT == 1 && p.topk_k <= kTopKMax && p.topk_k <= p.N && !I[GEMM_I_relu] &&
                    L->topk_idx_raw != 0 && L->topk_probs_raw != 0 && p.topk_part != nullptr && p.topk_cnt != nullptr &&
                    !(op.p[GEMM_P_topk_part] & VQA_EXT_TAG) && !(op.p[GEMM_P_topk_cnt] & VQA_EXT_TAG),
                VQA_E_INVALID, "gemm: the fused top-k epilogue needs 16-bit operands, an fp32 output without residual, BN = 128, "
                               "MT = 1, k <= 8 and its scratch buffers");
    L->epi = 6;
  }

  // shared-memory plan: one CTA per SM (persistent): rings + epilogue staging + bias table + barriers <= 227 KB
  const int stage_bytes = epi_stage_bytes(L->epi, sf);
  const int fixed_bytes = 1024 + stage_bytes + 4 * kBiasTable + 8 * (2 * kMaxASlots + 2 * kMaxBSlots + 4 + kMaxEpiWarps) + 16 +
                          4 * VQA_MAX_TAPS + 16 * VQA_MAX_GROUPS + (sf > 1 ? kXchgBytes : 0);
  int budget = I[GEMM_I_smem_budget];
  if (budget <= 0) {   // experiment switch: cap the CTA's total shared memory (KB) so CTAs of other kernels can co-reside
    static const int cap_kb = std::getenv("VQA_GEMM_SMEM_KB") ? std::atoi(std::getenv("VQA_GEMM_SMEM_KB")) : 0;
    if (cap_kb > 0 && cap_kb * 1024 > fixed_bytes + 32 * 1024) budget = cap_kb * 1024 - fixed_bytes;
  }
  if (budget <= 0 || budget > 227 * 1024 - fixed_bytes) budget = 227 * 1024 - fixed_bytes;
  const long long b_all = static_cast<long long>(p.k_chunks) * p.b_slot_bytes;
  p.b_resident = (p.n_tiles == 1 && b_all <= 96 * 1024 && b_all + 2LL * p.a_slot_bytes <= budget) ? 1 : 0;
  if (p.b_resident) {
    int s = static_cast<int>((budget - b_all) / p.a_slot_bytes);
    p.a_slots = s < 2 ? 2 : (s > kMaxASlots ? kMaxASlots : s);
    p.b_slots = 1;
  } else if (lockstep) {
    int s = budget / (p.a_slot_bytes + p.b_slot_bytes);
    s = s < 2 ? 2 : (s > kMaxASlots ? kMaxASlots : s);
    p.a_slots = p.b_slots = s;
  } else {
    // window mode: 3 windows in flight when they are cheap, the rest of the budget to the weight ring
    p.a_slots = (3 * p.a_slot_bytes + 4 * p.b_slot_bytes <= budget) ? 3 : 2;
    int s = (budget - p.a_slots * p.a_slot_bytes) / p.b_slot_bytes;
    p.b_slots = s < 2 ? 2 : (s > kMaxBSlots ? kMaxBSlots : s);
  }
  const long long b_bytes = p.b_resident ? b_all : static_cast<long long>(p.b_slots) * p.b_slot_bytes;
  L->smem = static_cast<size_t>(fixed_bytes) + static_cast<size_t>(p.a_slots) * p.a_slot_bytes + static_cast<size_t>(b_bytes);
  VQA_REQUIRE(L->smem <= 227 * 1024, VQA_E_INVALID, "gemm: shared memory budget exceeded");

  // tensor maps (only for non-external operands: A and W always live in the arenas)
  VQA_REQUIRE(!(op.p[GEMM_P_a0] & VQA_EXT_TAG) && !(op.p[GEMM_P_b] & VQA_EXT_TAG) && !(op.p[GEMM_P_a1] & VQA_EXT_TAG),
              VQA_E_INVALID, "gemm: A/B operands must be arena buffers");
  int rc = encode_2d(&L->mapA0, tf32, op.p[GEMM_P_a0], I[GEMM_I_a0_rows], I[GEMM_I_a0_cols], I[GEMM_I_a0_ld],
                     p.box_rows, p.row_bytes, "gemm A0");
  if (rc) return rc;
  if (uses_a1) {
    VQA_REQUIRE(op.p[GEMM_P_a1] != 0, VQA_E_INVALID, "gemm: group references A1 but it is null");
    rc = encode_2d(&L->mapA1, tf32, op.p[GEMM_P_a1], I[GEMM_I_a1_rows], I[GEMM_I_a1_cols], I[GEMM_I_a1_ld],
                   p.box_rows, p.row_bytes, "gemm A1");
    if (rc) return rc;
  } else {
    L->mapA1 = L->mapA0;
  }
  rc = encode_2d(&L->mapB, tf32, op.p[GEMM_P_b], I[GEMM_I_Npad], I[GEMM_I_Ktot], I[GEMM_I_Ktot], pair ? n_mma / 2 : n_mma,
                 p.row_bytes, "gemm B");
  if (rc) return rc;

  p.ldo = I[GEMM_I_ldo];
  p.ldr = I[GEMM_I_ldr];
  p.relu = I[GEMM_I_relu];
  p.round_tf32 = I[GEMM_I_round_tf32];
  p.mask_en = I[GEMM_I_mask_en];
  p.mP = I[GEMM_I_mP] > 0 ? I[GEMM_I_mP] : 1;
  p.mRPI = I[GEMM_I_mRPI] > 0 ? I[GEMM_I_mRPI] : 1;
  p.mH = I[GEMM_I_mH];
  p.mW = I[GEMM_I_mW];
  auto magic = [](int d, uint32_t* m, uint32_t* sh) {   // n / d == umulhi(n, m) >> sh for 0 <= n < 2^31, d >= 2
    int k = 0;
    while ((1LL << k) < d) ++k;
    *m = static_cast<uint32_t>((1ULL << (31 + k)) / static_cast<unsigned long long>(d) + 1ULL);
    *sh = static_cast<uint32_t>(k - 1);
  };
  p.rpi_magic = p.rpi_shift = p.mp_magic = p.mp_shift = 0;
  if (p.mask_en) {
    VQA_REQUIRE(p.mP >= 2 && p.mRPI >= 2 && p.M < (1 << 30), VQA_E_INVALID, "gemm: pad-mask grid out of range");
    magic(p.mRPI, &p.rpi_magic, &p.rpi_shift);
    magic(p.mP, &p.mp_magic, &p.mp_shift);
    for (long long n = 0; n < (1LL << 31); n += 104729) {   // spot check of the division identity
      const uint32_t q = static_cast<uint32_t>((static_cast<unsigned long long>(n) * p.rpi_magic) >> 32) >> p.rpi_shift;
      VQA_REQUIRE(q == static_cast<uint32_t>(n / p.mRPI), VQA_E_INVALID, "gemm: division magic failed");
    }
  }
  p.bias = reinterpret_cast<const float*>(op.p[GEMM_P_bias]);
  VQA_REQUIRE(p.bias == nullptr || (reinterpret_cast<uintptr_t>(p.bias) & 15) == 0, VQA_E_ALIGN,
              "gemm: bias must be 16-byte aligned");
  p.dbg = reinterpret_cast<long long*>(op.p[GEMM_P_dbg]);
  p.sums = reinterpret_cast<float*>(op.p[GEMM_P_sums]);
  p.ld_sums = p.N;
  VQA_REQUIRE(p.sums == nullptr || (!(op.p[GEMM_P_sums] & VQA_EXT_TAG) && p.out_dtype != 1 && sf == 1 && !pool && p.tiles_per_img == 0),
              VQA_E_INVALID, "gemm: slab column sums need a 16-bit output and the linear M tiling");
  L->out_raw = op.p[GEMM_P_out];
  L->res_raw = op.p[GEMM_P_res];
  VQA_REQUIRE(L->out_raw != 0, VQA_E_INVALID, "gemm: null output");
  L->bn = bn;
  L->threads = sf > 1 ? kSfThreads : kThreads;
  const int tiles = p.m_tiles * p.n_tiles;
  int sms = num_sms(device);
  if (I[GEMM_I_max_ctas] > 0 && I[GEMM_I_max_ctas] < sms) sms = I[GEMM_I_max_ctas];   // tests: force many tiles per CTA
  // Walkers (CTAs, or CTA pairs) = the fewest that finish in the same number of rounds: 226 pair tiles on 74 pairs take 4
  // rounds whether 74 or 57 pairs walk them, and the SMs left free run other kernels (the other compute lanes' batches:
  // measured 198.4k -> 203.1k pairs/s with three lanes, single stream unchanged).
  static const bool balance = std::getenv("VQA_NO_GRID_BALANCE") == nullptr;
  auto walkers_for = [&](int units) {
    units = units > 0 ? units : 1;
    if (tiles <= units) return tiles;
    const int rounds = (tiles + units - 1) / units;
    return balance ? (tiles + rounds - 1) / rounds : units;
  };
  if (pair) {
    L->grid = dim3(2 * walkers_for(sms / 2), 1, 1);
  } else {
    L->grid = dim3(walkers_for(sms), 1, 1);
  }

  L->out_external = (L->out_raw & VQA_EXT_TAG) != 0;
  L->mapOut = L->mapA0;
  L->mapRes = L->mapA0;
  L->mapOutLast = L->mapA0;
  if (pool) {
    VQA_REQUIRE(!has_res && p.out_dtype == 0 && !L->out_external, VQA_E_INVALID,
                "gemm: the pooled output is a bf16 arena buffer without residual");
  } else {
    VQA_REQUIRE(sf == 1 || !L->out_external, VQA_E_INVALID, "gemm: shift-fused outputs are arena buffers");
    if (!L->out_external) {
      // shift-fused kernels: the last 32-row slab of a tile stores only its complete rows
      rc = encode_box32(&L->mapOut, p.out_dtype == 1, L->out_raw, p.M, p.N, p.ldo, "gemm output");
      if (rc) return rc;
      if (sf > 1) {
        rc = encode_box32(&L->mapOutLast, p.out_dtype == 1, L->out_raw, p.M, p.N, p.ldo, "gemm output (last slab)",
                          32 - (sf - 1) * p.sf_step);
        if (rc) return rc;
      }
    }
    if (has_res) {
      VQA_REQUIRE(!(L->res_raw & VQA_EXT_TAG), VQA_E_INVALID, "gemm: the residual must be an arena buffer");
      rc = encode_box32(&L->mapRes, p.res_dtype == 1, L->res_raw, p.M, p.N, p.ldr, "gemm residual");
      if (rc) return rc;
    }
  }
  L->fn = pick_kernel(bn, p.MT, tf32, L->epi, p.row_bytes, pair, sf);
  VQA_REQUIRE(L->fn != nullptr, VQA_E_INVALID, "gemm: no kernel instantiation for this BN/MT/dtype/epilogue");
  VQA_CUDA_OK(cudaFuncSetAttribute(reinterpret_cast<const void*>(L->fn), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   227 * 1024));
  return VQA_OK;
}

int gemm_run(const void* storage, const uint64_t* ext, int n_ext, cudaStream_t stream) {
  const GemmLaunch* L = reinterpret_cast<const GemmLaunch*>(storage);
  GemmParams p = L->prm;
  p.out = reinterpret_cast<void*>(vqa_resolve(L->out_raw, ext, n_ext));
  p.res = reinterpret_cast<const void*>(vqa_resolve(L->res_raw, ext, n_ext));
  VQA_REQUIRE(p.out != nullptr, VQA_E_INVALID, "gemm: unresolved external output");
  if (p.topk_k > 0) {
    p.topk_idx = reinterpret_cast<long long*>(vqa_resolve(L->topk_idx_raw, ext, n_ext));
    p.topk_probs = reinterpret_cast<float*>(vqa_resolve(L->topk_probs_raw, ext, n_ext));
    VQA_REQUIRE(p.topk_idx != nullptr && p.topk_probs != nullptr, VQA_E_INVALID, "gemm: unresolved top-k outputs");
  }
  if (L->out_external) {   // caller-owned output: encode its store map for this call (host-only work, graph-capturable)
    CUtensorMap mo;
    int rc = encode_box32(&mo, p.out_dtype == 1, reinterpret_cast<uint64_t>(p.out), p.M, p.N, p.ldo, "gemm output");
    if (rc) return rc;
    VQA_CUDA_OK(vqa_launch_cluster(L->fn, L->grid, dim3(L->threads), L->smem, stream, L->pair ? 2 : 1, L->mapA0, L->mapA1, L->mapB,
                                   mo, L->mapRes, L->mapOutLast, p));
  } else {
    VQA_CUDA_OK(vqa_launch_cluster(L->fn, L->grid, dim3(L->threads), L->smem, stream, L->pair ? 2 : 1, L->mapA0, L->mapA1, L->mapB,
                                   L->mapOut, L->mapRes, L->mapOutLast, p));
  }
  VQA_LAUNCH_OK("gemm_tap_kernel");
  return VQA_OK;
}

const char* gemm_kernel_name(const void* storage) {
  const GemmLaunch* L = reinterpret_cast<const GemmLaunch*>(storage);
  static thread_local char name[64];
  const int sf = static_cast<int>((L->prm.idesc >> 17) & 63u) * 8 / L->bn;
  snprintf(name, sizeof(name), "gemm_tap_kernel<%d,%d,%s,e%d%s%s%s>", L->bn, L->prm.MT,
           L->prm.is_tf32 ? "tf32" : (((L->prm.idesc >> 7) & 7u) == 0u ? "f16" : "bf16"), L->epi,
           L->prm.row_bytes == 32 ? ",row32" : "", L->pair ? ",pair" : "", sf == 3 ? ",sf3" : sf == 2 ? ",sf2" : "");
  return name;
}
