// C ABI of libvqa_b200.so: plans (immutable op lists with pre-encoded tensor maps), error
// reporting and launch accounting.  See include/vqa_b200.h for the contract.
#include <atomic>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "common.cuh"

// implemented in gemm_tcgen05.cu / kernels_misc.cu
int gemm_launch_bytes();
int gemm_prepare(const VqaOp& op, void* storage, int device);
int gemm_run(const void* storage, const uint64_t* ext, int n_ext, cudaStream_t stream);
const char* gemm_kernel_name(const void* storage);
int stem_launch_bytes();
int stem_prepare(const VqaOp& op, void* storage, int device);
int stem_run(const void* storage, const uint64_t* ext, int n_ext, cudaStream_t stream);
int chain_launch_bytes();
int chain_prepare(const VqaOp& op, void* storage, int device);
int chain_run(const void* storage, const uint64_t* ext, int n_ext, cudaStream_t stream);
int run_misc_op(const VqaOp& op, const uint64_t* ext, int n_ext, cudaStream_t st);
const char* misc_kernel_name(int kind);

namespace {
thread_local std::string g_error;
std::atomic<uint64_t> g_launches{0};

struct FieldCount { int ni, np, nf; };
const FieldCount kFields[VQA_OP_KIND_MAX] = {
    {0, 0, 0},
    {INGEST_NI, INGEST_NP, INGEST_NF},
    {GEMM_NI, GEMM_NP, GEMM_NF},
    {MAXPOOL_NI, MAXPOOL_NP, MAXPOOL_NF},
    {SE_SQUEEZE_NI, SE_SQUEEZE_NP, SE_SQUEEZE_NF},
    {SE_EXCITE_NI, SE_EXCITE_NP, SE_EXCITE_NF},
    {SPATIAL_MAP_NI, SPATIAL_MAP_NP, SPATIAL_MAP_NF},
    {SCALE_RELAYOUT_NI, SCALE_RELAYOUT_NP, SCALE_RELAYOUT_NF},
    {EMBED_NI, EMBED_NP, EMBED_NF},
    {LAYERNORM_NI, LAYERNORM_NP, LAYERNORM_NF},
    {SELF_ATTN_NI, SELF_ATTN_NP, SELF_ATTN_NF},
    {CROSS_ATTN_NI, CROSS_ATTN_NP, CROSS_ATTN_NF},
    {POOL_GATE_LN_NI, POOL_GATE_LN_NP, POOL_GATE_LN_NF},
    {SOFTMAX_TOPK_NI, SOFTMAX_TOPK_NP, SOFTMAX_TOPK_NF},
    {MASK_PREP_NI, MASK_PREP_NP, MASK_PREP_NF},
    {GRID_TO_NCHW_NI, GRID_TO_NCHW_NP, GRID_TO_NCHW_NF},
    {COPY_ROWS_NI, COPY_ROWS_NP, COPY_ROWS_NF},
    {STAGE_TAIL_NI, STAGE_TAIL_NP, STAGE_TAIL_NF},
    {SPLIT_TF32_NI, SPLIT_TF32_NP, SPLIT_TF32_NF},
    {STEM_POOL_NI, STEM_POOL_NP, STEM_POOL_NF},
    {MLP_CHAIN_NI, MLP_CHAIN_NP, MLP_CHAIN_NF},
    {ATTN_CHUNKED_NI, ATTN_CHUNKED_NP, ATTN_CHUNKED_NF},
};
static_assert(MLP_CHAIN_NP <= VQA_OP_NP, "VqaOp.p too small for the chain op");
static_assert(GEMM_NI <= VQA_OP_NI, "VqaOp.i too small for the gemm op");
static_assert(POOL_GATE_LN_NP <= VQA_OP_NP, "VqaOp.p too small");
}  // namespace

void vqa_set_error(const std::string& msg) { g_error = msg; }
bool vqa_pdl_enabled() {
  static const bool on = std::getenv("VQA_NO_PDL") == nullptr;
  return on;
}

void vqa_count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

struct VqaPlan {
  int device = 0;
  std::vector<VqaOp> ops;
  std::vector<void*> gemm;   // per op: prepared GemmLaunch / StemLaunch (64-byte aligned) or nullptr
  std::atomic_flag busy = ATOMIC_FLAG_INIT;   // set while a host thread enqueues this plan (events / side stream are per plan)
  bool has_side = false;     // some op runs on lane 1
  cudaStream_t side = nullptr;
  static constexpr int kEvents = 16;   // fork / join edges of one run (cycled)
  cudaEvent_t events[kEvents] = {};
  ~VqaPlan() {
    for (void* g : gemm)
      if (g) std::free(g);
    for (cudaEvent_t e : events)
      if (e) cudaEventDestroy(e);
    if (side) cudaStreamDestroy(side);
  }
};

extern "C" {

int vqa_abi_version(void) { return VQA_ABI_VERSION; }

const char* vqa_last_error(void) { return g_error.c_str(); }

uint64_t vqa_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int vqa_device_check(int device) {
  cudaDeviceProp prop;
  VQA_CUDA_OK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    vqa_set_error(std::string("device ") + prop.name + " is compute capability " + std::to_string(prop.major) + "." +
                  std::to_string(prop.minor) + "; libvqa_b200 is built for sm_100a only");
    return VQA_E_UNSUPPORTED;
  }
  return VQA_OK;
}

int vqa_op_num_fields(int kind, int* n_i, int* n_p, int* n_f) {
  VQA_REQUIRE(kind >= 1 && kind < VQA_OP_KIND_MAX, VQA_E_INVALID, "unknown op kind");
  if (n_i) *n_i = kFields[kind].ni;
  if (n_p) *n_p = kFields[kind].np;
  if (n_f) *n_f = kFields[kind].nf;
  return VQA_OK;
}

int vqa_plan_create(const VqaOp* ops, int32_t n_ops, int32_t device, VqaPlan** out) {
  VQA_REQUIRE(ops != nullptr && out != nullptr && n_ops > 0, VQA_E_INVALID, "vqa_plan_create: null argument");
  *out = nullptr;
  int rc = vqa_device_check(device);
  if (rc) return rc;
  // tensor maps, streams and function attributes belong to `device`; the caller's current device is restored on return
  struct DeviceGuard {
    int prev = -1;
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
  } guard;
  VQA_CUDA_OK(cudaGetDevice(&guard.prev));
  if (guard.prev == device) guard.prev = -1; else VQA_CUDA_OK(cudaSetDevice(device));
  VqaPlan* plan = new (std::nothrow) VqaPlan();
  VQA_REQUIRE(plan != nullptr, VQA_E_INVALID, "out of host memory");
  plan->device = device;
  plan->ops.assign(ops, ops + n_ops);
  plan->gemm.assign(n_ops, nullptr);
  for (int k = 0; k < n_ops; ++k) {
    const VqaOp& op = plan->ops[k];
    if (op.kind < 1 || op.kind >= VQA_OP_KIND_MAX) {
      vqa_set_error("op " + std::to_string(k) + ": unknown kind " + std::to_string(op.kind));
      delete plan;
      return VQA_E_INVALID;
    }
    if (op.kind == VQA_OP_GEMM || op.kind == VQA_OP_STEM_POOL || op.kind == VQA_OP_MLP_CHAIN) {   // ops with prepared launches (tensor maps encoded once)
      const bool is_gemm = op.kind == VQA_OP_GEMM, is_stem = op.kind == VQA_OP_STEM_POOL;
      void* st = nullptr;
      const size_t bytes = (static_cast<size_t>(is_gemm ? gemm_launch_bytes() : is_stem ? stem_launch_bytes() : chain_launch_bytes()) + 63) / 64 * 64;
      if (posix_memalign(&st, 64, bytes) != 0) {
        vqa_set_error("out of host memory");
        delete plan;
        return VQA_E_INVALID;
      }
      std::memset(st, 0, bytes);
      plan->gemm[k] = st;
      rc = is_gemm ? gemm_prepare(op, st, device) : is_stem ? stem_prepare(op, st, device) : chain_prepare(op, st, device);
      if (rc) {
        vqa_set_error("op " + std::to_string(k) + ": " + g_error);
        delete plan;
        return rc;
      }
    }
  }
  int edges = 0;
  for (const VqaOp& op : plan->ops) {
    plan->has_side |= (op.lane & 1) != 0;
    edges += (op.lane & VQA_LANE_JOIN) != 0;
  }
  if (edges + 2 > VqaPlan::kEvents) {
    vqa_set_error("too many lane joins in one plan");
    delete plan;
    return VQA_E_INVALID;
  }
  if (plan->has_side) {
    bool ok = cudaStreamCreateWithFlags(&plan->side, cudaStreamNonBlocking) == cudaSuccess;
    for (int e = 0; ok && e < VqaPlan::kEvents; ++e)
      ok = cudaEventCreateWithFlags(&plan->events[e], cudaEventDisableTiming) == cudaSuccess;
    if (!ok) {
      vqa_set_error("could not create the side stream / events");
      delete plan;
      return VQA_E_CUDA;
    }
  }
  *out = plan;
  return VQA_OK;
}

int vqa_plan_run_range(const VqaPlan* plan, int32_t first, int32_t last, const uint64_t* ext, int32_t n_ext,
                       void* stream) {
  VQA_REQUIRE(plan != nullptr, VQA_E_INVALID, "vqa_plan_run: null plan");
  const int n = static_cast<int>(plan->ops.size());
  VQA_REQUIRE(first >= 0 && last <= n && first <= last, VQA_E_INVALID, "vqa_plan_run: bad op range");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  // A plan owns its fork / join events and its side stream: two host threads must not enqueue the same plan at the same
  // time (use one plan per slot).  Detected, not serialised: the second caller gets an error instead of a silent race.
  VqaPlan* mut = const_cast<VqaPlan*>(plan);
  if (mut->busy.test_and_set(std::memory_order_acquire)) {
    vqa_set_error("vqa_plan_run: this plan is being enqueued by another thread (plans are not re-entrant; use one plan per stream)");
    return VQA_E_INVALID;
  }
  struct RunGuard {
    VqaPlan* plan;
    int prev = -1;
    ~RunGuard() {
      if (prev >= 0) cudaSetDevice(prev);
      plan->busy.clear(std::memory_order_release);
    }
  } guard{mut};
  {   // kernels and events of this plan live on plan->device, whatever the calling thread's current device is
    int cur = -1;
    VQA_CUDA_OK(cudaGetDevice(&cur));
    if (cur != plan->device) {
      VQA_CUDA_OK(cudaSetDevice(plan->device));
      guard.prev = cur;
    }
  }
  // Whole-plan runs put lane-1 ops (bit 0 of VqaOp.lane) on the plan's side stream.  The first lane-1 op of a
  // run forks (the side stream waits for everything the caller's stream holds so far); an op with
  // VQA_LANE_JOIN set waits for all work issued so far on the OTHER lane before it starts; the end of the plan
  // joins the side stream back.  Partial ranges run serially on the caller's stream.
  static const bool lanes_off = std::getenv("VQA_NO_LANES") != nullptr;   // A/B switch: everything on the caller's stream
  const bool two_lanes = plan->has_side && first == 0 && last == n && !lanes_off;
  bool side_used = false;
  int ev = 0;
  auto edge = [&](cudaStream_t from, cudaStream_t to) -> int {
    cudaEvent_t e = plan->events[ev];
    ev = (ev + 1) % VqaPlan::kEvents;
    VQA_CUDA_OK(cudaEventRecord(e, from));
    VQA_CUDA_OK(cudaStreamWaitEvent(to, e, 0));
    return VQA_OK;
  };
  for (int k = first; k < last; ++k) {
    const VqaOp& op = plan->ops[k];
    cudaStream_t s = st;
    if (two_lanes) {
      const bool side = (op.lane & 1) != 0, join = (op.lane & VQA_LANE_JOIN) != 0;
      if (side && !side_used) {
        if (int rc = edge(st, plan->side)) return rc;
        side_used = true;
      } else if (join && side_used) {
        if (int rc = side ? edge(st, plan->side) : edge(plan->side, st)) return rc;
      }
      if (side) s = plan->side;
    }
    int rc = (op.kind == VQA_OP_GEMM) ? gemm_run(plan->gemm[k], ext, n_ext, s)
             : (op.kind == VQA_OP_STEM_POOL) ? stem_run(plan->gemm[k], ext, n_ext, s)
             : (op.kind == VQA_OP_MLP_CHAIN) ? chain_run(plan->gemm[k], ext, n_ext, s) : run_misc_op(op, ext, n_ext, s);
    if (rc) {
      vqa_set_error("op " + std::to_string(k) + ": " + g_error);
      return rc;
    }
  }
  if (side_used) {   // the caller's stream must observe everything the side lane did
    if (int rc = edge(plan->side, st)) return rc;
  }
  return VQA_OK;
}

int vqa_plan_run(const VqaPlan* plan, const uint64_t* ext, int32_t n_ext, void* stream) {
  VQA_REQUIRE(plan != nullptr, VQA_E_INVALID, "vqa_plan_run: null plan");
  return vqa_plan_run_range(plan, 0, static_cast<int32_t>(plan->ops.size()), ext, n_ext, stream);
}

int vqa_plan_num_launches(const VqaPlan* plan) { return plan ? static_cast<int>(plan->ops.size()) : 0; }

int vqa_plan_op_kernel_name(const VqaPlan* plan, int32_t op, char* buf, int32_t buflen) {
  VQA_REQUIRE(plan != nullptr && buf != nullptr && buflen > 0, VQA_E_INVALID, "null argument");
  VQA_REQUIRE(op >= 0 && op < static_cast<int32_t>(plan->ops.size()), VQA_E_INVALID, "op index out of range");
  const char* name = plan->ops[op].kind == VQA_OP_GEMM ? gemm_kernel_name(plan->gemm[op])
                     : plan->ops[op].kind == VQA_OP_STEM_POOL ? "stem_pool_kernel"
                     : plan->ops[op].kind == VQA_OP_MLP_CHAIN ? "mlp_chain_kernel" : misc_kernel_name(plan->ops[op].kind);
  std::strncpy(buf, name, static_cast<size_t>(buflen) - 1);
  buf[buflen - 1] = 0;
  return VQA_OK;
}

void vqa_plan_destroy(VqaPlan* plan) { delete plan; }

}  // extern "C"
