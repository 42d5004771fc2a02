// hmpc_capi.cu — host side of libhector_mpc_b200.so: the C-ABI declared in include/hector_mpc_b200.h.
//
// Part 1 re-exports the reference's boundary (convexMPC_interface.h:39-43) on top of a one-robot
// context; part 2 is the batched interface.  There is no CPU solve path in this library.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <unistd.h>

#include <chrono>
#include <cstddef>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <atomic>
#include <condition_variable>
#include <cstring>
#include <ctime>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/hector_mpc_b200.h"
#include "hmpc_device.cuh"

static_assert(sizeof(update_data_t) == 3016, "update_data_t must match convexMPC_interface.h:19-37");
static_assert(sizeof(problem_setup) == 16, "problem_setup must match convexMPC_interface.h:11-17");

namespace {

thread_local std::string g_err;

bool cuda_fail(cudaError_t e, const char* what)
{
  if (e == cudaSuccess) return false;
  g_err = std::string(what) + ": " + cudaGetErrorString(e);
  return true;
}
#define CK(call)                          \
  do {                                    \
    if (cuda_fail((call), #call)) return HMPC_ERR_CUDA; \
  } while (0)

// Small host worker pool for the byte-shuffling around the GPU call (packing records, widening results).
// Workers spin briefly after a job (a control loop calling at 200 Hz+ keeps them hot), then sleep.
class HostPool {
 public:
  explicit HostPool(int nworkers)
  {
    for (int i = 0; i < nworkers; i++) workers_.emplace_back([this, i] { run(i); });
  }
  ~HostPool()
  {
    {
      std::lock_guard<std::mutex> lk(m_);
      stop_ = true;
      gen_++;
    }
    cv_.notify_all();
    for (auto& t : workers_) t.join();
  }
  int size() const { return (int)workers_.size() + 1; }
  // run fn(part, nparts) on nparts = size() threads (the caller takes part 0); returns when all are done
  void parallel(const std::function<void(int, int)>& fn)
  {
    const int np = size();
    if (np == 1) { fn(0, 1); return; }
    fn_ = &fn;
    pending_.store(np - 1, std::memory_order_release);
    {
      std::lock_guard<std::mutex> lk(m_);
      gen_++;
    }
    cv_.notify_all();
    fn(0, np);
    while (pending_.load(std::memory_order_acquire) != 0) std::this_thread::yield();  // the parts are equal-sized: a short wait
  }

 private:
  void run(int idx)
  {
    unsigned seen = 0;
    for (;;) {
      // spin ~50 us for the next generation, then block
      bool got = false;
      const auto t0 = std::chrono::steady_clock::now();
      while (std::chrono::steady_clock::now() - t0 < std::chrono::microseconds(50)) {
        if (gen_relaxed() != seen) { got = true; break; }
      }
      if (!got) {
        std::unique_lock<std::mutex> lk(m_);
        cv_.wait(lk, [&] { return gen_ != seen; });
      }
      {
        std::lock_guard<std::mutex> lk(m_);
        seen = gen_;
        if (stop_) return;
      }
      (*fn_)(idx + 1, size());
      pending_.fetch_sub(1, std::memory_order_acq_rel);
    }
  }
  unsigned gen_relaxed()
  {
    std::lock_guard<std::mutex> lk(m_);
    return gen_;
  }
  std::vector<std::thread> workers_;
  std::mutex m_;
  std::condition_variable cv_;
  unsigned gen_ = 0;
  bool stop_ = false;
  const std::function<void(int, int)>* fn_ = nullptr;
  std::atomic<int> pending_{0};
};

constexpr int NCHUNK = 4;  // the host-buffer path pipelines pack / H2D / solve / D2H over this many chunks

struct ClassCfg {
  int nb_hi, nb_cap, qmax, threads, smem, grid_cap, variant, tcap;
  hmpc::Layout L;
};

}  // namespace

struct hmpc_ctx {
  int device = 0, max_batch = 0, horizon = 0, rec_stride = 0, sm_count = 0;
  problem_setup setup{};
  ClassCfg cls[3];
  int ncls = 0;
  unsigned char* d_rec = nullptr;
  unsigned char* d_out = nullptr;  // host-buffer path: per chunk [wrench floats | status ints], contiguous
  int* d_status = nullptr;         // scratch status (assembly hook)
  int* d_counts = nullptr;         // [NCHUNK][2] class list lengths
  int* d_lists = nullptr;          // [NCHUNK][2][max_batch] class lists (host-built, host-buffer path)
  int* d_cls = nullptr;            // [NCHUNK][2 parities x 4 lengths | class-1 list | class-2 list] (device-resident path)
  unsigned tick[NCHUNK] = {0, 0, 0, 0};  // calls per slot: parity of the list lengths in use
  unsigned char* h_rec = nullptr;  // pinned
  unsigned char* h_out = nullptr;  // pinned mirror of d_out
  unsigned char* d_states = nullptr;  // hmpc_state_t staging of hmpc_solve_batch_states (row f-1)
  unsigned char* h_states = nullptr;  // pinned
  int* h_cls = nullptr;            // pinned [NCHUNK][4 + 3*max_batch]: host-built class counts + lists (host-buffer path)
  cudaStream_t stream = nullptr;   // chunk 0 / single-robot stream
  cudaStream_t xstream[3] = {nullptr, nullptr, nullptr};  // further chunks of the pipelined host path
  HostPool* pool = nullptr;        // helper threads for packing / widening (large batches only)
  int max_iter = 500;  // same cap as the reference's nWSR (SolverMPC.cpp:584)
  // multi-GPU (one process per GPU, batch sharded): NCCL communicator + double-buffered float results for the gather
  void* nccl = nullptr;            // ncclComm_t
  int shard_rank = 0, shard_world = 1;
  float* shard_buf[2] = {nullptr, nullptr};   // [max_batch][12N] this rank's results of tick t / t+1
  float* shard_out = nullptr;      // where the kernels of the current sharded tick also store float results (else null)
  unsigned shard_tick = 0;
  bool shard_used = false;         // the in-place chain stored this tick's floats (else the staged path ran)
  cudaStream_t gstream = nullptr;  // the gather runs here, behind `solved`, beside the next tick
  cudaEvent_t solved = nullptr, gathered[2] = {nullptr, nullptr};
  int* d_ws = nullptr;             // [max_batch][WS_STATE_INTS] working sets of the previous tick (closed-loop warm start)
  int warm_start = 1;              // hmpc_rollout_device proposes them to the next tick (HMPC_WARM_START=0: cold start every tick)
  int lockstep = 1;                // waves of a multi-wave launch start together (HMPC_LOCKSTEP=0: free-running, for A/B runs)
  double kappa_max = 1.5e5;  // conditioning limit of the fp64 sweep inversion (HMPC_KAPPA_MAX; see the kernel's stage 5)
  int block_min = 2;     // later rounds need at least this many entering rows (HMPC_BLOCK_MIN, A/B knob)
  int block_rounds = 4;  // block start of the active-set stage (HMPC_BLOCK_ROUNDS=0: plain dual iteration, for A/B runs)
  // caller-owned host buffers registered with hmpc_pin_host_buffer: hmpc_solve_batch lets the kernels read the
  // reference records from them and write results to them in place (no packing, no staging copies, no widening)
  struct Pin { char* base; size_t bytes; };   // what the caller asked for
  struct Run { uintptr_t lo, hi; };           // page runs actually registered with CUDA (arrays may share pages)
  std::vector<Pin> pins;
  std::vector<Run> runs;
  bool pinned(const void* p, size_t bytes) const
  {
    const char* q = static_cast<const char*>(p);
    for (const Pin& r : pins)
      if (q >= r.base && q + bytes <= r.base + r.bytes) return true;
    return false;
  }
};

namespace {

// kernel variants <threads, min CTAs/SM, fixed horizon (0 = runtime), size class>
//   0/1: horizon 10 fixed at compile time (class 0: 4 warps, class 1: 8 warps)
//   10 + 5*cls + b: runtime horizon, b-th entry of {64, 128, 192, 256, 384} threads
#define HMPC_FOR_VARIANT(V, X)                   \
  switch (V) {                                   \
    case 0: X(128, 7, 10, 0); break;             \
    case 1: X(256, 2, 10, 1); break;             \
    case 10: X(64, 8, 0, 0); break;              \
    case 11: X(128, 6, 0, 0); break;             \
    case 12: X(192, 3, 0, 0); break;             \
    case 13: X(256, 2, 0, 0); break;             \
    case 14: X(384, 1, 0, 0); break;             \
    case 15: X(64, 8, 0, 1); break;              \
    case 16: X(128, 6, 0, 1); break;             \
    case 17: X(192, 3, 0, 1); break;             \
    case 18: X(256, 2, 0, 1); break;             \
    default: X(384, 1, 0, 1); break;             \
  }
const int kBucketThreads[5] = {64, 128, 192, 256, 384};

cudaError_t prep_class(ClassCfg& c, int* occ)
{
  cudaError_t e = cudaSuccess;
  // The attribute is per kernel instantiation and process-wide, and several contexts (other horizons, the
  // reference-style global context) share the runtime-horizon instantiations: always raise it to the device's opt-in
  // maximum instead of this context's carve-up, so no context can lower it under another's launches.
#define HMPC_PREP(NT, MB, NF, CL)                                                                       \
  {                                                                                                    \
    auto k = hmpc::hmpc_solve_kernel<NT, MB, NF, CL>;                                                  \
    e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);              \
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(occ, k, NT, c.smem);       \
  }
  HMPC_FOR_VARIANT(c.variant, HMPC_PREP)
#undef HMPC_PREP
  return e;
}

// programmatic dependent launch for the device-resident chain (classification -> class 0 -> class 1 -> class 2):
// every kernel of the chain may become resident while its predecessor drains and waits (griddepcontrol.wait) before it
// reads what the predecessor wrote.  HMPC_PDL=0 switches back to plain stream order.
bool pdl_enabled()
{
  static const bool on = !(getenv("HMPC_PDL") && atoi(getenv("HMPC_PDL")) == 0);
  return on;
}

template <typename... KArgs, typename... Args>
cudaError_t launch_chain(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl, Args... args)
{
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, args...);
}

cudaError_t launch_class(const ClassCfg& c, const hmpc::KernelArgs& ka, int grid, cudaStream_t st, bool pdl = false)
{
  cudaError_t e = cudaSuccess;
#define HMPC_LAUNCH(NT, MB, NF, CL) \
  e = launch_chain(hmpc::hmpc_solve_kernel<NT, MB, NF, CL>, dim3(grid), dim3(NT), (size_t)c.smem, st, pdl, ka);
  HMPC_FOR_VARIANT(c.variant, HMPC_LAUNCH)
#undef HMPC_LAUNCH
  return e != cudaSuccess ? e : cudaGetLastError();
}

int build_classes(hmpc_ctx* c)
{
  const int N = c->horizon;
  // class 0: at most N blocks of 6 variables (e.g. any single-support schedule); class 1: up to 2N.
  // Working-set overflow in class 0 escalates to class 1.
  // class 2 = class 1's size with as many working-set slots as one SM's shared memory holds (1 CTA/SM): reached only
  // by escalation from class 1 (massively degenerate optima, e.g. all contact forces at zero).
  c->ncls = 3;
  for (int i = 0; i < 3; i++) {
    ClassCfg& k = c->cls[i];
    if (i == 2) {
      // class 2: class 1's size, every row may be active; no H^-1 a_j cache (its primal steps go through a full product)
      k = c->cls[1];
      const int n = 6 * k.nb_cap;
      if (c->cls[1].qmax >= n) { c->ncls = 2; break; }  // class 1 already holds every row
      k.qmax = n;
      k.tcap = 0;
      if (N == 10) {  // the runtime-layout instantiation of the same shape (the fixed one folds class 1's layout)
        k.variant = 18;
        k.threads = 256;
      }
      k.L = hmpc::make_layout(N, k.nb_cap, k.qmax, c->rec_stride, k.threads / 32, 0);
      while (k.L.total > 226 * 1024 && k.qmax > c->cls[1].qmax) {
        k.qmax -= 4;
        k.L = hmpc::make_layout(N, k.nb_cap, k.qmax, c->rec_stride, k.threads / 32, 0);
      }
      if (k.qmax <= c->cls[1].qmax) { c->ncls = 2; break; }
      k.smem = k.L.total;
      int occ = 0;
      if (cuda_fail(prep_class(k, &occ), "kernel attribute/occupancy (class 2)")) return HMPC_ERR_CUDA;
      if (occ < 1) { g_err = "class-2 kernel does not fit on this device"; return HMPC_ERR_CUDA; }
      k.grid_cap = occ * c->sm_count;
      break;
    }
    k.nb_cap = hmpc::class_nb_cap(N, i);
    k.nb_hi = k.nb_cap;
    const int warps = hmpc::class_warps(N, i);
    int bucket = 0;
    while (bucket < 4 && kBucketThreads[bucket] < 32 * warps) bucket++;
    if (kBucketThreads[bucket] < 32 * warps) { g_err = "horizon too long for the built kernel variants"; return HMPC_ERR_ARG; }
    if (N == 10) {
      k.variant = i;
      k.threads = (i == 0) ? 128 : 256;
    } else {
      k.variant = 10 + 5 * i + bucket;
      k.threads = kBucketThreads[bucket];
    }
    k.qmax = hmpc::class_qmax(N, i);
    k.tcap = hmpc::class_tcap(N, i);
    k.L = hmpc::make_layout(N, k.nb_cap, k.qmax, c->rec_stride, k.threads / 32, k.tcap);
    k.smem = k.L.total;
    int occ = 0;
    if (cuda_fail(prep_class(k, &occ), "kernel attribute/occupancy (is this an sm_100a device?)")) return HMPC_ERR_CUDA;
    if (occ < 1) { g_err = "kernel does not fit on this device"; return HMPC_ERR_CUDA; }
    k.grid_cap = occ * c->sm_count;
  }
  return HMPC_OK;
}

hmpc::KernelArgs base_args(const hmpc_ctx* c, const void* d_records, int B, float* d_wrench, int* d_status)
{
  hmpc::KernelArgs ka{};
  ka.records = static_cast<const unsigned char*>(d_records);
  ka.rec_stride = c->rec_stride;
  ka.batch = B;
  ka.horizon = c->horizon;
  ka.dt = c->setup.dt;
  ka.f_max = c->setup.f_max;
  ka.max_iter = c->max_iter;
  ka.tol_kkt = 1e-9;
  ka.tol_dep = 1e-11;
  ka.block_rounds = c->block_rounds;
  ka.block_min = c->block_min;
  ka.kappa_max = c->kappa_max;
  ka.wrench = d_wrench;
  ka.status = d_status;
  return ka;
}

}  // namespace

// ---------------------------------------------------------------------------------------------------
// records
// ---------------------------------------------------------------------------------------------------
HMPC_EXTERNC size_t hmpc_record_bytes(int horizon)
{
  if (horizon < 1 || horizon > 18) return 0;
  size_t b = (size_t)(54 + 12 * horizon) * 4 + (size_t)2 * horizon;
  return (b + 15) / 16 * 16;
}

HMPC_EXTERNC int hmpc_pack_records(const update_data_t* in, int n, int horizon, void* out)
{
  const size_t stride = hmpc_record_bytes(horizon);
  if (!in || !out || n < 0 || stride == 0) { g_err = "hmpc_pack_records: bad argument"; return HMPC_ERR_ARG; }
  unsigned char* o = static_cast<unsigned char*>(out);
  for (int i = 0; i < n; i++, o += stride) {
    const update_data_t& u = in[i];
    if (i + 2 < n) {  // the live bytes of a record are ~11 scattered cache lines of 47: fetch ahead
      const char* nx = reinterpret_cast<const char*>(&in[i + 2]);
      for (int off = 0; off < (42 + 12 * horizon) * 4; off += 64) __builtin_prefetch(nx + off);
      __builtin_prefetch(nx + offsetof(update_data_t, Alpha_K));
      __builtin_prefetch(nx + offsetof(update_data_t, gait));
    }
    float* f = reinterpret_cast<float*>(o);
    memcpy(f, u.p, 42 * 4);  // p v q w r joint_angles yaw weights are contiguous in update_data_t
    memcpy(f + 42, u.Alpha_K, 48);
    memcpy(f + 54, u.traj, (size_t)48 * horizon);
    unsigned char* g = o + (size_t)(54 + 12 * horizon) * 4;
    memcpy(g, u.gait, (size_t)2 * horizon);
    memset(g + 2 * horizon, 0, stride - ((size_t)(54 + 12 * horizon) * 4 + 2 * horizon));
  }
  return HMPC_OK;
}

// ---------------------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------------------
HMPC_EXTERNC const char* hmpc_last_error(void) { return g_err.c_str(); }

// ---------------------------------------------------------------------------------------------------
// multi-GPU (SURVEY.md 8e): one process per GPU, contiguous batch slices, identical kernels, no data-path collective;
// ONE ncclAllGather of the float results when a consumer needs the whole batch on every device.  NCCL is looked up at
// run time (libnccl.so.2 — the copy the process already holds when PyTorch is loaded), so the library has no link
// dependency on it and single-GPU users never touch it.
// ---------------------------------------------------------------------------------------------------
struct Id128 { char b[128]; };  // ncclUniqueId, passed by value
namespace {
struct NcclApi {
  void* h = nullptr;
  int (*GetUniqueId)(void*) = nullptr;
  int (*CommInitRank)(void**, int, Id128, int) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
}  // namespace
namespace {
NcclApi g_nccl;
bool nccl_load()
{
  if (g_nccl.h) return true;
  void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!h) { g_err = std::string("NCCL not found: ") + dlerror(); return false; }
  g_nccl.GetUniqueId = reinterpret_cast<int (*)(void*)>(dlsym(h, "ncclGetUniqueId"));
  g_nccl.CommInitRank = reinterpret_cast<int (*)(void**, int, Id128, int)>(dlsym(h, "ncclCommInitRank"));
  g_nccl.AllGather = reinterpret_cast<int (*)(const void*, void*, size_t, int, void*, cudaStream_t)>(dlsym(h, "ncclAllGather"));
  g_nccl.CommDestroy = reinterpret_cast<int (*)(void*)>(dlsym(h, "ncclCommDestroy"));
  g_nccl.GetErrorString = reinterpret_cast<const char* (*)(int)>(dlsym(h, "ncclGetErrorString"));
  if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllGather || !g_nccl.CommDestroy) {
    g_err = "NCCL library lacks ncclGetUniqueId / ncclCommInitRank / ncclAllGather / ncclCommDestroy";
    return false;
  }
  g_nccl.h = h;
  return true;
}
bool nccl_fail(int rc, const char* what)
{
  if (rc == 0) return false;
  g_err = std::string(what) + ": " + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "NCCL error");
  return true;
}
void shard_release(hmpc_ctx* c)
{
  if (c->nccl && g_nccl.CommDestroy) g_nccl.CommDestroy(c->nccl);
  c->nccl = nullptr;
  for (int i = 0; i < 2; i++) {
    if (c->shard_buf[i]) cudaFree(c->shard_buf[i]);
    if (c->gathered[i]) cudaEventDestroy(c->gathered[i]);
    c->shard_buf[i] = nullptr;
    c->gathered[i] = nullptr;
  }
  if (c->solved) cudaEventDestroy(c->solved);
  if (c->gstream) cudaStreamDestroy(c->gstream);
  c->solved = nullptr;
  c->gstream = nullptr;
}
}  // namespace

HMPC_EXTERNC int hmpc_shard_unique_id(void* id128)
{
  if (!id128) { g_err = "hmpc_shard_unique_id: null argument"; return HMPC_ERR_ARG; }
  if (!nccl_load()) return HMPC_ERR_CUDA;
  if (nccl_fail(g_nccl.GetUniqueId(id128), "ncclGetUniqueId")) return HMPC_ERR_CUDA;
  return HMPC_OK;
}

HMPC_EXTERNC int hmpc_shard_init(hmpc_ctx* c, int rank, int world, const void* id128)
{
  if (!c || !id128 || world < 1 || rank < 0 || rank >= world) { g_err = "hmpc_shard_init: bad argument"; return HMPC_ERR_ARG; }
  if (c->nccl) { g_err = "hmpc_shard_init: context already belongs to a shard group"; return HMPC_ERR_ARG; }
  if (!nccl_load()) return HMPC_ERR_CUDA;
  CK(cudaSetDevice(c->device));
  Id128 id;
  memcpy(id.b, id128, 128);
  if (nccl_fail(g_nccl.CommInitRank(&c->nccl, world, id, rank), "ncclCommInitRank")) return HMPC_ERR_CUDA;
  c->shard_rank = rank;
  c->shard_world = world;
  const size_t nw = (size_t)12 * c->horizon;
  CK(cudaStreamCreateWithFlags(&c->gstream, cudaStreamNonBlocking));
  CK(cudaEventCreateWithFlags(&c->solved, cudaEventDisableTiming));
  for (int i = 0; i < 2; i++) {
    CK(cudaMalloc(&c->shard_buf[i], (size_t)c->max_batch * nw * sizeof(float)));
    CK(cudaEventCreateWithFlags(&c->gathered[i], cudaEventDisableTiming));
  }
  return HMPC_OK;
}

HMPC_EXTERNC int hmpc_solve_batch_sharded(hmpc_ctx* c, const update_data_t* in_local, int B_local, double* wrench_local,
                                          int* status_local, float* d_all)
{
  if (!c || !c->nccl) { g_err = "hmpc_solve_batch_sharded: call hmpc_shard_init first"; return HMPC_ERR_ARG; }
  if (B_local < 1 || B_local > c->max_batch) { g_err = "hmpc_solve_batch_sharded: every rank needs 1 <= B_local <= capacity"; return HMPC_ERR_ARG; }
  CK(cudaSetDevice(c->device));
  const int par = (int)(c->shard_tick++ & 1u);
  const size_t nw = (size_t)12 * c->horizon;
  if (d_all) {
    // this tick's kernels also leave float results in shard_buf[par]; the gather that last read it (two ticks ago)
    // must be done before they overwrite it — a stream-side wait, the host does not block
    CK(cudaStreamWaitEvent(c->stream, c->gathered[par], 0));
    c->shard_out = c->shard_buf[par];
  }
  const int rc = hmpc_solve_batch(c, in_local, B_local, wrench_local, status_local);
  const bool staged = d_all && c->shard_out && !c->shard_used;
  c->shard_out = nullptr;
  if (rc != HMPC_OK && rc != HMPC_ERR_NOT_CONVERGED) return rc;
  if (d_all) {
    if (staged) {
      // the staged host path did not run the in-place chain: put the float results on the device for the gather
      std::vector<float> tmp((size_t)B_local * nw);
      for (size_t i = 0; i < tmp.size(); i++) tmp[i] = (float)wrench_local[i];
      CK(cudaMemcpyAsync(c->shard_buf[par], tmp.data(), tmp.size() * sizeof(float), cudaMemcpyHostToDevice, c->stream));
      CK(cudaStreamSynchronize(c->stream));
      CK(cudaEventRecord(c->solved, c->stream));
    }
    c->shard_used = false;
    // the path's ONE collective: every rank's slice of float wrenches to every device, beside the next tick
    CK(cudaStreamWaitEvent(c->gstream, c->solved, 0));
    if (nccl_fail(g_nccl.AllGather(c->shard_buf[par], d_all, (size_t)B_local * nw, /* ncclFloat32 */ 7, c->nccl, c->gstream), "ncclAllGather"))
      return HMPC_ERR_CUDA;
    CK(cudaEventRecord(c->gathered[par], c->gstream));
  }
  return rc;
}

HMPC_EXTERNC int hmpc_shard_wait(hmpc_ctx* c)
{
  if (!c || !c->nccl) { g_err = "hmpc_shard_wait: call hmpc_shard_init first"; return HMPC_ERR_ARG; }
  CK(cudaSetDevice(c->device));
  CK(cudaStreamSynchronize(c->gstream));
  return HMPC_OK;
}

HMPC_EXTERNC void hmpc_destroy(hmpc_ctx* c)
{
  if (!c) return;
  cudaSetDevice(c->device);
  for (const hmpc_ctx::Run& r : c->runs) cudaHostUnregister(reinterpret_cast<void*>(r.lo));
  c->runs.clear();
  c->pins.clear();
  if (c->d_rec) cudaFree(c->d_rec);
  if (c->d_out) cudaFree(c->d_out);
  if (c->d_status) cudaFree(c->d_status);
  if (c->d_counts) cudaFree(c->d_counts);
  if (c->d_lists) cudaFree(c->d_lists);
  if (c->d_cls) cudaFree(c->d_cls);
  shard_release(c);
  if (c->d_ws) cudaFree(c->d_ws);
  if (c->d_states) cudaFree(c->d_states);
  if (c->h_states) cudaFreeHost(c->h_states);
  if (c->h_rec) cudaFreeHost(c->h_rec);
  if (c->h_out) cudaFreeHost(c->h_out);
  if (c->h_cls) cudaFreeHost(c->h_cls);
  delete c->pool;
  if (c->stream) cudaStreamDestroy(c->stream);
  for (int i = 0; i < 3; i++)
    if (c->xstream[i]) cudaStreamDestroy(c->xstream[i]);
  delete c;
}

HMPC_EXTERNC hmpc_ctx* hmpc_create(int max_batch, int horizon, int device)
{
  if (max_batch < 1 || horizon < 1 || horizon > HMPC_MAX_HORIZON) {
    g_err = "hmpc_create: need max_batch >= 1 and 1 <= horizon <= 16";
    return nullptr;
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= device || device < 0) {
    g_err = "hmpc_create: no usable CUDA device (this library has no CPU path)";
    return nullptr;
  }
  hmpc_ctx* c = new hmpc_ctx;
  c->device = device;
  c->max_batch = max_batch;
  c->horizon = horizon;
  c->rec_stride = (int)hmpc_record_bytes(horizon);
  c->setup.dt = 0.04f;
  c->setup.mu = 0.25f;
  c->setup.f_max = 500.f;
  c->setup.horizon = horizon;
  cudaDeviceProp prop{};
  bool bad = cuda_fail(cudaSetDevice(device), "cudaSetDevice") ||
             cuda_fail(cudaGetDeviceProperties(&prop, device), "cudaGetDeviceProperties");
  if (!bad && prop.major != 10) {
    g_err = "hmpc_create: kernels are built for sm_100a only; device is sm_" + std::to_string(prop.major) +
            std::to_string(prop.minor);
    bad = true;
  }
  if (!bad) {
    c->sm_count = prop.multiProcessorCount;
    const size_t nw = (size_t)12 * horizon;
    bad = cuda_fail(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking), "cudaStreamCreate") ||
          cuda_fail(cudaStreamCreateWithFlags(&c->xstream[0], cudaStreamNonBlocking), "cudaStreamCreate") ||
          cuda_fail(cudaStreamCreateWithFlags(&c->xstream[1], cudaStreamNonBlocking), "cudaStreamCreate") ||
          cuda_fail(cudaStreamCreateWithFlags(&c->xstream[2], cudaStreamNonBlocking), "cudaStreamCreate") ||
          cuda_fail(cudaMalloc(&c->d_rec, (size_t)max_batch * c->rec_stride), "cudaMalloc records") ||
          cuda_fail(cudaMalloc(&c->d_out, (size_t)max_batch * (nw * 4 + 4 + 40)), "cudaMalloc results") ||
          cuda_fail(cudaMalloc(&c->d_counts, NCHUNK * 4 * sizeof(int)), "cudaMalloc counts") ||
          cuda_fail(cudaMalloc(&c->d_lists, (size_t)NCHUNK * (4 + 3 * (size_t)max_batch) * sizeof(int)), "cudaMalloc lists") ||
          cuda_fail(cudaMalloc(&c->d_ws, (size_t)max_batch * hmpc::WS_STATE_INTS * sizeof(int)), "cudaMalloc working sets") ||
          cuda_fail(cudaMemset(c->d_ws, 0, (size_t)max_batch * hmpc::WS_STATE_INTS * sizeof(int)), "cudaMemset working sets") ||
          cuda_fail(cudaMalloc(&c->d_cls, (size_t)NCHUNK * (8 + 2 * (size_t)max_batch) * sizeof(int)), "cudaMalloc class lists") ||
          cuda_fail(cudaMemset(c->d_cls, 0, (size_t)NCHUNK * (8 + 2 * (size_t)max_batch) * sizeof(int)), "cudaMemset class lists") ||
          cuda_fail(cudaMalloc(&c->d_status, (size_t)max_batch * 4), "cudaMalloc status") ||
          cuda_fail(cudaMalloc(&c->d_states, (size_t)max_batch * sizeof(hmpc_state_t)), "cudaMalloc states") ||
          cuda_fail(cudaMallocHost(&c->h_states, (size_t)max_batch * sizeof(hmpc_state_t)), "cudaMallocHost states") ||
          cuda_fail(cudaMallocHost(&c->h_rec, (size_t)max_batch * c->rec_stride), "cudaMallocHost records") ||
          cuda_fail(cudaMallocHost(&c->h_out, (size_t)max_batch * (nw * 4 + 4 + 40)), "cudaMallocHost results") ||
          cuda_fail(cudaMallocHost(&c->h_cls, (size_t)NCHUNK * (4 + 3 * (size_t)max_batch) * sizeof(int)), "cudaMallocHost lists") ||
          build_classes(c) != HMPC_OK;
  }
  if (!bad) {
    const char* br = getenv("HMPC_BLOCK_ROUNDS");
    if (br) c->block_rounds = atoi(br);
    if (const char* bm = getenv("HMPC_BLOCK_MIN")) c->block_min = atoi(bm);
    if (const char* km = getenv("HMPC_KAPPA_MAX")) c->kappa_max = atof(km);
    const char* ls = getenv("HMPC_LOCKSTEP");
    if (ls) c->lockstep = atoi(ls);
    const char* wm = getenv("HMPC_WARM_START");
    if (wm) c->warm_start = atoi(wm);
  }
  if (!bad && max_batch >= 256) {
    const char* e = getenv("HMPC_HOST_THREADS");
    int nt = e ? atoi(e) : 4;
    const int hw = (int)std::thread::hardware_concurrency();
    if (hw > 0 && nt > hw) nt = hw;
    if (nt > 1) c->pool = new HostPool(nt - 1);
  }
  if (bad) {
    std::string keep = g_err;
    hmpc_destroy(c);
    g_err = keep;
    return nullptr;
  }
  return c;
}

HMPC_EXTERNC int hmpc_set_problem(hmpc_ctx* c, const problem_setup* s)
{
  if (!c || !s) { g_err = "hmpc_set_problem: null argument"; return HMPC_ERR_ARG; }
  if (s->horizon != c->horizon) { g_err = "hmpc_set_problem: horizon differs from the context's"; return HMPC_ERR_ARG; }
  c->setup = *s;
  return HMPC_OK;
}

namespace {
long long* g_dbg_clk = nullptr;  // profiling hook (hmpc_debug_set_clock_buffer)
// classification pre-pass + one launch per class, all enqueued on `st`
int enqueue_solve(hmpc_ctx* c, const void* d_records, int B, float* d_wrench32, double* d_wrench64, int* d_status,
                  cudaStream_t st, int slot = 0, float* d_tau = nullptr, int* d_ws = nullptr, int ws_shift = 0, bool ws_read = false,
                  const update_data_t* raw = nullptr)
{
  if (B > c->max_batch) { g_err = "batch exceeds the context's capacity"; return HMPC_ERR_ARG; }
  CK(cudaSetDevice(c->device));
  // per slot: [2 parities][4 list lengths], then the lists of class 1 and class 2.  No classification kernel: the
  // class-0 launch runs over every instance and hands the ones with more stance blocks than it holds to class 1's list.
  int* base = c->d_cls + (size_t)slot * (8 + 2 * (size_t)c->max_batch);
  const int par = (c->tick[slot]++) & 1;
  int* counts = base + 4 * par;
  int* counts_next = base + 4 * (par ^ 1);
  int* lists = base + 8 - (size_t)c->max_batch;  // lists + i * max_batch is class i's list, i = 1, 2
  const bool pdl = pdl_enabled();
  for (int i = 0; i < c->ncls; i++) {
    const ClassCfg& k = c->cls[i];
    hmpc::KernelArgs ka = base_args(c, d_records, B, d_wrench32, d_status);
    ka.wrench64 = d_wrench64;
    ka.raw_records = reinterpret_cast<const unsigned char*>(raw);
    ka.tau = d_tau;
    ka.warm_start = (d_ws && ws_read) ? 1 : 0;
    ka.ws_state = d_ws;
    ka.ws_shift = ws_shift;
    ka.list = (i == 0) ? nullptr : lists + (size_t)i * c->max_batch;
    ka.split_nb = (i == 0) ? k.nb_hi : -1;
    ka.counts_next = (i == 0) ? counts_next : nullptr;
    // arrival counter of class 0's wave barrier: the 4th length slot, which the chain does not use.  (Class 1 runs free:
    // its instances differ more in length, and waiting for the slowest of every wave cost more than lockstep gained — A/B at
    // 8192 mixed robots +6 %, horizon 5 -20 %, horizon 16 -5 %.)
    ka.wave_sync = (c->lockstep && i == 0) ? reinterpret_cast<unsigned*>(counts + 3) : nullptr;
    ka.counts = counts;
    ka.cls = i;
    ka.esc_list = (i + 1 < c->ncls) ? lists + (size_t)(i + 1) * c->max_batch : nullptr;
    ka.nb_cap = k.nb_cap;
    ka.qmax = k.qmax;
    ka.tcap = k.tcap;
    ka.L = k.L;
    ka.dbg_clk = g_dbg_clk;
    const int grid = B < k.grid_cap ? B : k.grid_cap;
    CK(launch_class(k, ka, grid, st, pdl));
  }
  return HMPC_OK;
}
}  // namespace

namespace {
// Host-buffer path: the host has the contact tables in hand while it packs, so it builds the class lists itself
// (same rule as hmpc_classify_kernel) and launches only the non-empty classes — no classification kernel, no
// empty launches.  Working-set overflow cannot escalate here; the caller re-runs such a chunk through enqueue_solve.
void classify_host(const hmpc_ctx* c, const unsigned char* gait0, size_t gait_stride, int nb, int* blockbuf)
{
  int* counts = blockbuf;
  int* lists = blockbuf + 4;
  counts[0] = counts[1] = counts[2] = counts[3] = 0;
  const int N = c->horizon;
  for (int i = 0; i < nb; i++) {
    int k = 0;
    for (int e = 0; e < 2 * N; e++) {
      const float ub = c->setup.f_max * (float)gait0[(size_t)i * gait_stride + e];
      k += !(ub < 0.0001f && ub > -0.0001f);
    }
    const int cl = (k <= c->cls[0].nb_hi) ? 0 : 1;
    lists[(size_t)cl * c->max_batch + counts[cl]++] = i;
  }
}

int enqueue_solve_hostlists(hmpc_ctx* c, const void* d_records, int nb, int* h_block, float* d_wrench32, int* d_status,
                            cudaStream_t st, int slot, float* d_tau, bool zero_copy, const update_data_t* raw = nullptr,
                            double* wrench64 = nullptr)
{
  int* d_block = c->d_lists + (size_t)slot * (4 + 3 * (size_t)c->max_batch);
  const int n0 = h_block[0], n1 = h_block[1];
  if (zero_copy) {
    d_block = h_block;  // pinned + mapped: the kernels read the lists over PCIe, no copy launch
  } else {
    // counts + class-0 list (+ class-1 list when it is not empty) in one copy
    const size_t ints = (n1 > 0) ? (size_t)4 + c->max_batch + n1 : (size_t)4 + n0;
    CK(cudaMemcpyAsync(d_block, h_block, ints * sizeof(int), cudaMemcpyHostToDevice, st));
  }
  for (int i = 0; i < 2; i++) {
    const int cnt = i == 0 ? n0 : n1;
    if (cnt == 0) continue;
    const ClassCfg& k = c->cls[i];
    hmpc::KernelArgs ka = base_args(c, d_records, nb, d_wrench32, d_status);
    ka.raw_records = reinterpret_cast<const unsigned char*>(raw);
    ka.wrench64 = wrench64;
    ka.tau = d_tau;
    ka.warm_start = 0;
    ka.list = d_block + 4 + (size_t)i * c->max_batch;
    ka.counts = d_block;
    ka.cls = i;
    ka.esc_list = nullptr;  // overflow is handled by the caller's retry
    ka.split_nb = -1;
    ka.nb_cap = k.nb_cap;
    ka.qmax = k.qmax;
    ka.tcap = k.tcap;
    ka.L = k.L;
    ka.dbg_clk = g_dbg_clk;
    const int grid = cnt < k.grid_cap ? cnt : k.grid_cap;
    CK(launch_class(k, ka, grid, st));
  }
  return HMPC_OK;
}
}  // namespace

// The kernels stage a record with a 1-D bulk copy (cp.async.bulk), whose global source must be 16-byte aligned: the record
// stride is a multiple of 16 by construction, the base pointer is the caller's (a sliced tensor view may not be).
static int check_device_records(const hmpc_ctx* c, const void* d_records, int B, const char* who)
{
  if (B > c->max_batch) { g_err = std::string(who) + ": batch exceeds the context's capacity"; return HMPC_ERR_ARG; }
  if (reinterpret_cast<uintptr_t>(d_records) & 15u) { g_err = std::string(who) + ": d_records must be 16-byte aligned"; return HMPC_ERR_ARG; }
  return HMPC_OK;
}

// profiling hook: device buffer [batch][32] of clock64() stage timestamps, or NULL to switch off
HMPC_EXTERNC void hmpc_debug_set_clock_buffer(long long* d_buf) { g_dbg_clk = d_buf; }

// fault-injection hook (tests): the next n host-buffer solves return HMPC_ERR_CUDA without touching the device — what a
// run-time CUDA failure looks like to the callers (the reference boundary's status path, tests/test_zzz_reference_status_path.py)
namespace { int g_fail_next_solves = 0; }
HMPC_EXTERNC void hmpc_debug_fail_next_solves(int n) { g_fail_next_solves = n; }

HMPC_EXTERNC int hmpc_launches_per_solve(const hmpc_ctx* c) { return c ? c->ncls : 0; }

// launch configuration of class `cls`: out[0..5] = threads, dynamic smem bytes, working-set capacity,
// resident-grid cap (CTAs), max blocks of 6 variables, sweep strip width
HMPC_EXTERNC int hmpc_class_config(const hmpc_ctx* c, int cls, int* out)
{
  if (!c || !out || cls < 0 || cls >= c->ncls) return HMPC_ERR_ARG;
  const ClassCfg& k = c->cls[cls];
  out[0] = k.threads; out[1] = k.smem; out[2] = k.qmax; out[3] = k.grid_cap; out[4] = k.nb_cap;
  out[5] = 8;  // sweep tile edge (8x8 mma.m8n8k4.f64 accumulator tiles)
  return HMPC_OK;
}

HMPC_EXTERNC int hmpc_solve_device(hmpc_ctx* c, const void* d_records, int B, float* d_wrench, int* d_status,
                                   void* stream)
{
  if (!c || !d_records || !d_wrench || !d_status || B < 0) { g_err = "hmpc_solve_device: bad argument"; return HMPC_ERR_ARG; }
  if (B == 0) return HMPC_OK;
  if (int rc = check_device_records(c, d_records, B, "hmpc_solve_device")) return rc;
  return enqueue_solve(c, d_records, B, d_wrench, nullptr, d_status, static_cast<cudaStream_t>(stream));
}

HMPC_EXTERNC int hmpc_solve_device_ex(hmpc_ctx* c, const void* d_records, int B, float* d_wrench, int* d_status,
                                      float* d_tau, void* stream)
{
  if (!c || !d_records || !d_wrench || !d_status || B < 0) { g_err = "hmpc_solve_device_ex: bad argument"; return HMPC_ERR_ARG; }
  if (B == 0) return HMPC_OK;
  if (int rc = check_device_records(c, d_records, B, "hmpc_solve_device_ex")) return rc;
  return enqueue_solve(c, d_records, B, d_wrench, nullptr, d_status, static_cast<cudaStream_t>(stream), 0, d_tau);
}

HMPC_EXTERNC int hmpc_assemble_device(hmpc_ctx* c, const void* d_records, int B, float* d_H, float* d_g,
                                      float* d_Fblk, float* d_lb, float* d_ub, void* stream)
{
  if (!c || !d_records || !d_H || !d_g || !d_Fblk || !d_lb || !d_ub || B < 0) {
    g_err = "hmpc_assemble_device: bad argument";
    return HMPC_ERR_ARG;
  }
  if (B == 0) return HMPC_OK;
  if (int rc = check_device_records(c, d_records, B, "hmpc_assemble_device")) return rc;
  CK(cudaSetDevice(c->device));
  const ClassCfg& k = c->cls[c->ncls - 1];
  hmpc::KernelArgs ka = base_args(c, d_records, B, nullptr, c->d_status);
  ka.list = nullptr;  // identity
  ka.split_nb = -1;
  ka.counts = c->d_counts;
  ka.cls = c->ncls - 1;
  ka.esc_list = nullptr;
  ka.nb_cap = k.nb_cap;
  ka.qmax = k.qmax;
  ka.tcap = k.tcap;
  ka.L = k.L;
  ka.dbg_H = d_H;
  ka.dbg_g = d_g;
  ka.dbg_F = d_Fblk;
  ka.dbg_lb = d_lb;
  ka.dbg_ub = d_ub;
  const int grid = B < k.grid_cap ? B : k.grid_cap;
  CK(launch_class(k, ka, grid, static_cast<cudaStream_t>(stream)));
  return HMPC_OK;
}

static int solve_batch_impl(hmpc_ctx* c, const update_data_t* in, const hmpc_state_t* sin, int B, double* wrench_out,
                            double* tau_out, int* status, double dtMPC = 0.0);

HMPC_EXTERNC int hmpc_solve_batch(hmpc_ctx* c, const update_data_t* in, int B, double* wrench_out, int* status)
{
  return solve_batch_impl(c, in, nullptr, B, wrench_out, nullptr, status);
}

HMPC_EXTERNC int hmpc_solve_batch_ex(hmpc_ctx* c, const update_data_t* in, int B, double* wrench_out, double* tau_out,
                                     int* status)
{
  return solve_batch_impl(c, in, nullptr, B, wrench_out, tau_out, status);
}

static_assert(sizeof(hmpc_state_t) == 352 && offsetof(hmpc_state_t, gait) == 39 * 8, "hmpc_state_t layout (hmpc_prepare_kernel)");

HMPC_EXTERNC int hmpc_prepare_device(hmpc_ctx* c, const hmpc_state_t* d_states, int B, double dtMPC, void* d_records,
                                     void* stream)
{
  if (!c || !d_states || !d_records || B < 0) { g_err = "hmpc_prepare_device: bad argument"; return HMPC_ERR_ARG; }
  if (B == 0) return HMPC_OK;
  CK(cudaSetDevice(c->device));
  hmpc::hmpc_prepare_kernel<<<(B + 63) / 64, 64, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const unsigned char*>(d_states), B, c->horizon, dtMPC,
      static_cast<unsigned char*>(d_records), c->rec_stride);
  CK(cudaGetLastError());
  return HMPC_OK;
}

HMPC_EXTERNC int hmpc_pin_host_buffer(hmpc_ctx* c, void* ptr, size_t bytes)
{
  if (!c || !ptr || bytes == 0) { g_err = "hmpc_pin_host_buffer: bad argument"; return HMPC_ERR_ARG; }
  if (c->pinned(ptr, bytes)) return HMPC_OK;
  CK(cudaSetDevice(c->device));
  // registration is page-granular and two small caller arrays may share a page: register only the page runs of
  // [ptr, ptr+bytes) that no earlier pin covers
  const uintptr_t PG = (uintptr_t)(sysconf(_SC_PAGESIZE) > 0 ? sysconf(_SC_PAGESIZE) : 4096);  // 64 KiB on some aarch64 hosts
  const uintptr_t lo = reinterpret_cast<uintptr_t>(ptr) & ~(PG - 1);
  const uintptr_t hi = (reinterpret_cast<uintptr_t>(ptr) + bytes + PG - 1) & ~(PG - 1);
  auto covered = [&](uintptr_t pg) {
    for (const hmpc_ctx::Run& r : c->runs)
      if (pg >= r.lo && pg < r.hi) return true;
    return false;
  };
  for (uintptr_t pg = lo; pg < hi;) {
    if (covered(pg)) { pg += PG; continue; }
    uintptr_t end = pg + PG;
    while (end < hi && !covered(end)) end += PG;
    void* base = reinterpret_cast<void*>(pg);
    {
      cudaError_t re = cudaHostRegister(base, end - pg, cudaHostRegisterMapped | cudaHostRegisterPortable);
      if (re == cudaErrorHostMemoryAlreadyRegistered) cudaGetLastError();  // registered by somebody else: usable as it is
      else if (cuda_fail(re, "cudaHostRegister")) return HMPC_ERR_CUDA;
    }
    void* dptr = nullptr;
    cudaError_t e = cudaHostGetDevicePointer(&dptr, base, 0);
    if (e != cudaSuccess || dptr != base) {  // the in-place mode hands host addresses to the kernels
      cudaHostUnregister(base);
      g_err = "hmpc_pin_host_buffer: this device cannot address registered host memory through the host pointer";
      return HMPC_ERR_CUDA;
    }
    c->runs.push_back({pg, end});
    pg = end;
  }
  c->pins.push_back({static_cast<char*>(ptr), bytes});
  return HMPC_OK;
}

HMPC_EXTERNC int hmpc_unpin_host_buffer(hmpc_ctx* c, void* ptr)
{
  if (!c || !ptr) { g_err = "hmpc_unpin_host_buffer: bad argument"; return HMPC_ERR_ARG; }
  size_t idx = c->pins.size();
  for (size_t i = 0; i < c->pins.size(); i++)
    if (c->pins[i].base == static_cast<char*>(ptr)) idx = i;
  if (idx == c->pins.size()) { g_err = "hmpc_unpin_host_buffer: pointer was not pinned through this context"; return HMPC_ERR_ARG; }
  CK(cudaSetDevice(c->device));
  CK(cudaStreamSynchronize(c->stream));
  for (int i = 0; i < 3; i++) CK(cudaStreamSynchronize(c->xstream[i]));
  c->pins.erase(c->pins.begin() + idx);
  // release the page runs no remaining pin touches
  for (size_t r = 0; r < c->runs.size();) {
    bool used = false;
    for (const hmpc_ctx::Pin& p : c->pins) {
      const uintptr_t a = reinterpret_cast<uintptr_t>(p.base), b = a + p.bytes;
      used |= (a < c->runs[r].hi && b > c->runs[r].lo);
    }
    if (used) { r++; continue; }
    CK(cudaHostUnregister(reinterpret_cast<void*>(c->runs[r].lo)));
    c->runs.erase(c->runs.begin() + r);
  }
  return HMPC_OK;
}

static_assert(sizeof(hmpc_rollout_t) == 80 && offsetof(hmpc_rollout_t, gait_offset) == 48, "hmpc_rollout_t layout (hmpc_advance_kernel)");

HMPC_EXTERNC int hmpc_rollout_device(hmpc_ctx* c, hmpc_state_t* d_states, hmpc_rollout_t* d_loop, int B, int ticks,
                                     double dtMPC, float* d_wrench_log, void* d_record_log, void* stream)
{
  if (!c || !d_states || !d_loop || B < 0 || B > c->max_batch || ticks < 1) {
    g_err = "hmpc_rollout_device: bad argument (null pointer, batch > capacity or ticks < 1)";
    return HMPC_ERR_ARG;
  }
  if (B == 0) return HMPC_OK;
  CK(cudaSetDevice(c->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t nw = (size_t)12 * c->horizon;
  float* dw = reinterpret_cast<float*>(c->d_out);  // the context's own result area is the loop's scratch
  int* ds = reinterpret_cast<int*>(c->d_out + (size_t)c->max_batch * nw * 4);
  for (int t = 0; t < ticks; t++) {
    int rc = hmpc_prepare_device(c, d_states, B, dtMPC, c->d_rec, st);
    if (rc != HMPC_OK) return rc;
    if (d_record_log)
      CK(cudaMemcpyAsync(static_cast<unsigned char*>(d_record_log) + (size_t)t * B * c->rec_stride, c->d_rec,
                         (size_t)B * c->rec_stride, cudaMemcpyDeviceToDevice, st));
    rc = enqueue_solve(c, c->d_rec, B, dw, nullptr, ds, st, 0, nullptr, c->warm_start ? c->d_ws : nullptr, 1, true);
    if (rc != HMPC_OK) return rc;
    hmpc::hmpc_advance_kernel<<<(B + 63) / 64, 64, 0, st>>>(reinterpret_cast<unsigned char*>(d_states),
                                                            reinterpret_cast<unsigned char*>(d_loop), B, c->horizon, dtMPC, dw, ds,
                                                            d_wrench_log ? d_wrench_log + (size_t)t * B * 12 : nullptr);
    CK(cudaGetLastError());
  }
  return HMPC_OK;
}

HMPC_EXTERNC int hmpc_reset_warm_start(hmpc_ctx* c, void* stream)
{
  if (!c) { g_err = "hmpc_reset_warm_start: null context"; return HMPC_ERR_ARG; }
  CK(cudaSetDevice(c->device));
  CK(cudaMemsetAsync(c->d_ws, 0, (size_t)c->max_batch * hmpc::WS_STATE_INTS * sizeof(int), static_cast<cudaStream_t>(stream)));
  return HMPC_OK;
}

static_assert(sizeof(hmpc_swing_t) == 72 && offsetof(hmpc_swing_t, first_swing) == 64, "hmpc_swing_t layout (hmpc_swing_kernel)");
static_assert(sizeof(hmpc_swing_cmd_t) == 232 && offsetof(hmpc_swing_cmd_t, swing) == 224, "hmpc_swing_cmd_t layout (hmpc_swing_kernel)");

HMPC_EXTERNC int hmpc_swing_device(hmpc_ctx* c, const hmpc_state_t* d_states, const hmpc_rollout_t* d_loop, const double* d_phase,
                                   hmpc_swing_t* d_swing, int B, double dt, double dtSwing, hmpc_swing_cmd_t* d_cmd, void* stream)
{
  if (!c || !d_states || !d_loop || !d_phase || !d_swing || !d_cmd || B < 0) { g_err = "hmpc_swing_device: bad argument"; return HMPC_ERR_ARG; }
  if (B == 0) return HMPC_OK;
  CK(cudaSetDevice(c->device));
  hmpc::hmpc_swing_kernel<<<(B + 63) / 64, 64, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const unsigned char*>(d_states), reinterpret_cast<const unsigned char*>(d_loop), d_phase,
      reinterpret_cast<unsigned char*>(d_swing), B, c->horizon, dt, dtSwing, reinterpret_cast<unsigned char*>(d_cmd));
  CK(cudaGetLastError());
  return HMPC_OK;
}

HMPC_EXTERNC int hmpc_solve_batch_states(hmpc_ctx* c, const hmpc_state_t* in, int B, double dtMPC, double* wrench_out,
                                         double* tau_out, int* status)
{
  return solve_batch_impl(c, nullptr, in, B, wrench_out, tau_out, status, dtMPC);
}

static int solve_batch_impl(hmpc_ctx* c, const update_data_t* in, const hmpc_state_t* sin, int B, double* wrench_out,
                            double* tau_out, int* status, double dtMPC)
{
  if (!c || (!in && !sin) || !wrench_out || B < 0 || B > c->max_batch) {
    g_err = "hmpc_solve_batch: bad argument (null pointer or batch > capacity)";
    return HMPC_ERR_ARG;
  }
  if (B == 0) return HMPC_OK;
  if (g_fail_next_solves > 0) {
    g_fail_next_solves--;
    g_err = "injected failure (hmpc_debug_fail_next_solves)";
    return HMPC_ERR_CUDA;
  }
  CK(cudaSetDevice(c->device));
  const size_t nw = (size_t)12 * c->horizon;
  // pipeline over chunks: the host packs chunk k+1 while the GPU copies/solves chunk k, and converts the
  // results of chunk k while later chunks are still in flight
  static const int nch_env = getenv("HMPC_CHUNKS") ? atoi(getenv("HMPC_CHUNKS")) : 0;
  int nch = B >= 512 ? 2 : 1;  // with helper threads packing is short: two chunks overlap copy-back with compute
  if (!c->pool) nch = B >= 512 ? NCHUNK : (B >= 128 ? 2 : 1);
  if (nch_env >= 1 && nch_env <= NCHUNK) nch = nch_env;
  static const bool trace = getenv("HMPC_TRACE") != nullptr;
  // zero-copy mode: the kernels read the packed records from, and write the results to, pinned host memory
  // directly (UVA-mapped), so a tick has no copy launches at all.  Measured on B200: 0.224 vs 0.243 ms per
  // 1024-robot tick; beyond ~1.5k robots the two-chunk copy pipeline wins (0.66 vs 0.80 ms at 4096) because packing
  // overlaps the kernels there.  HMPC_ZEROCOPY=0/1 forces a mode.
  static const int zc_env = getenv("HMPC_ZEROCOPY") ? atoi(getenv("HMPC_ZEROCOPY")) : -1;
  const bool zc = zc_env >= 0 ? (zc_env != 0) : (B <= 1536);
  if (zc && nch_env < 1) nch = 1;
  // in-place mode: records, wrenches and status all live in buffers the caller registered (hmpc_pin_host_buffer):
  // the kernels gather the live bytes of every update_data_t over PCIe and store double results where the caller
  // wants them — the call is host classification + launches + one synchronize
  if (in && zc_env != 0 && !c->pins.empty() && c->pinned(in, (size_t)B * sizeof(update_data_t)) &&
      c->pinned(wrench_out, (size_t)B * nw * sizeof(double)) && (!status || c->pinned(status, (size_t)B * sizeof(int)))) {
    // the device-resident chain on the caller's records: class 0 classifies on the way, overflow escalates on the device
    int* ds = status ? status : reinterpret_cast<int*>(c->h_out + (size_t)c->max_batch * nw * 4);
    float* dt_ = tau_out ? reinterpret_cast<float*>(c->h_out + (size_t)c->max_batch * (nw * 4 + 4)) : nullptr;
    int rc = enqueue_solve(c, nullptr, B, c->shard_out, wrench_out, ds, c->stream, 0, dt_, nullptr, 0, false, in);
    if (rc != HMPC_OK) return rc;
    if (c->shard_out) {
      CK(cudaEventRecord(c->solved, c->stream));
      c->shard_used = true;
    }
    CK(cudaStreamSynchronize(c->stream));
    bool all_ok = true;
    for (int i = 0; i < B; i++) all_ok &= (HMPC_STATUS_CODE(ds[i]) == 0);
    if (tau_out)
      for (int i = 0; i < B * 10; i++) tau_out[i] = (double)dt_[i];
    if (!all_ok) { g_err = "hmpc_solve_batch: at least one instance did not reach a KKT point (see status[])"; return HMPC_ERR_NOT_CONVERGED; }
    return HMPC_OK;
  }
  double tr[4 * NCHUNK + 2];
  int ntr = 0;
  auto now = []() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec * 1e6 + ts.tv_nsec * 1e-3; };
  if (trace) tr[ntr++] = now();
  int lo[NCHUNK + 1];
  for (int k = 0; k <= nch; k++) lo[k] = (int)((long long)B * k / nch);
  cudaStream_t sts[NCHUNK] = {c->stream, c->xstream[0], c->xstream[1], c->xstream[2]};
  for (int k = 0; k < nch; k++) {
    const int b0 = lo[k], nb = lo[k + 1] - lo[k];
    if (nb == 0) continue;
    int rc = HMPC_OK;
    if (sin) {
      // row f-1: ship the 352-byte states and build the packed records on the device
      const size_t sb = sizeof(hmpc_state_t);
      memcpy(c->h_states + (size_t)b0 * sb, sin + b0, (size_t)nb * sb);
      if (trace) tr[ntr++] = now();
      if (!zc) CK(cudaMemcpyAsync(c->d_states + (size_t)b0 * sb, c->h_states + (size_t)b0 * sb, (size_t)nb * sb, cudaMemcpyHostToDevice, sts[k]));
      rc = hmpc_prepare_device(c, reinterpret_cast<const hmpc_state_t*>((zc ? c->h_states : c->d_states) + (size_t)b0 * sb), nb, dtMPC,
                               c->d_rec + (size_t)b0 * c->rec_stride, sts[k]);
      if (rc != HMPC_OK) return rc;
    } else {
      if (c->pool && nb >= 128) {
        c->pool->parallel([&](int part, int nparts) {
          const int p0 = (int)((long long)nb * part / nparts), p1 = (int)((long long)nb * (part + 1) / nparts);
          hmpc_pack_records(in + b0 + p0, p1 - p0, c->horizon, c->h_rec + (size_t)(b0 + p0) * c->rec_stride);
        });
      } else {
        rc = hmpc_pack_records(in + b0, nb, c->horizon, c->h_rec + (size_t)b0 * c->rec_stride);
      }
      if (rc != HMPC_OK) return rc;
      if (trace) tr[ntr++] = now();
      if (!zc)
        CK(cudaMemcpyAsync(c->d_rec + (size_t)b0 * c->rec_stride, c->h_rec + (size_t)b0 * c->rec_stride,
                           (size_t)nb * c->rec_stride, cudaMemcpyHostToDevice, sts[k]));
    }
    const size_t ooff = (size_t)b0 * (nw * 4 + 4 + 40), obytes = (size_t)nb * (nw * 4 + 4 + (tau_out ? 40 : 0));
    unsigned char* obase = zc ? c->h_out : c->d_out;
    float* dw = reinterpret_cast<float*>(obase + ooff);
    int* ds = reinterpret_cast<int*>(obase + ooff + (size_t)nb * nw * 4);
    float* dt_ = tau_out ? reinterpret_cast<float*>(obase + ooff + (size_t)nb * (nw * 4 + 4)) : nullptr;
    const unsigned char* rbase = (zc && !sin) ? c->h_rec : c->d_rec;
    int* hblk = c->h_cls + (size_t)k * (4 + 3 * (size_t)c->max_batch);
    if (sin) classify_host(c, sin[b0].gait, sizeof(hmpc_state_t), nb, hblk);
    else classify_host(c, in[b0].gait, sizeof(update_data_t), nb, hblk);
    rc = enqueue_solve_hostlists(c, rbase + (size_t)b0 * c->rec_stride, nb, hblk, dw, ds, sts[k], k, dt_, zc);
    if (rc != HMPC_OK) return rc;
    if (!zc) CK(cudaMemcpyAsync(c->h_out + ooff, c->d_out + ooff, obytes, cudaMemcpyDeviceToHost, sts[k]));
    if (trace) tr[ntr++] = now();
  }
  bool all_ok = true;
  for (int k = 0; k < nch; k++) {
    const int b0 = lo[k], nb = lo[k + 1] - lo[k];
    if (nb == 0) continue;
    CK(cudaStreamSynchronize(sts[k]));
    if (trace) tr[ntr++] = now();
    const size_t ooff = (size_t)b0 * (nw * 4 + 4 + 40);
    {  // working-set overflow (rare, massively degenerate optima): redo the chunk through the escalating device path
      const int* hs = reinterpret_cast<const int*>(c->h_out + ooff + (size_t)nb * nw * 4);
      bool overflow = false;
      for (int i = 0; i < nb; i++) overflow |= (HMPC_STATUS_CODE(hs[i]) == hmpc::ST_WS_CAP);
      if (overflow) {
        unsigned char* obase = zc ? c->h_out : c->d_out;
        float* dw = reinterpret_cast<float*>(obase + ooff);
        int* ds = reinterpret_cast<int*>(obase + ooff + (size_t)nb * nw * 4);
        float* dt_ = tau_out ? reinterpret_cast<float*>(obase + ooff + (size_t)nb * (nw * 4 + 4)) : nullptr;
        const unsigned char* rbase = (zc && !sin) ? c->h_rec : c->d_rec;
        int rc = enqueue_solve(c, rbase + (size_t)b0 * c->rec_stride, nb, dw, nullptr, ds, sts[k], k, dt_);
        if (rc != HMPC_OK) return rc;
        if (!zc)
          CK(cudaMemcpyAsync(c->h_out + ooff, c->d_out + ooff, (size_t)nb * (nw * 4 + 4 + (tau_out ? 40 : 0)),
                             cudaMemcpyDeviceToHost, sts[k]));
        CK(cudaStreamSynchronize(sts[k]));
      }
    }
    if (tau_out) {
      const float* ht = reinterpret_cast<const float*>(c->h_out + ooff + (size_t)nb * (nw * 4 + 4));
      for (int i = 0; i < nb * 10; i++) tau_out[(size_t)b0 * 10 + i] = (double)ht[i];
    }
    const float* src = reinterpret_cast<const float*>(c->h_out + ooff);
    const int* hst = reinterpret_cast<const int*>(c->h_out + ooff + (size_t)nb * nw * 4);
    double* dst = wrench_out + (size_t)b0 * nw;
    const size_t tot = (size_t)nb * nw;
    if (c->pool && nb >= 128) {
      c->pool->parallel([&](int part, int nparts) {
        const size_t i0 = tot * part / nparts, i1 = tot * (part + 1) / nparts;
        for (size_t i = i0; i < i1; i++) dst[i] = (double)src[i];
      });
    } else {
      for (size_t i = 0; i < tot; i++) dst[i] = (double)src[i];
    }
    for (int i = 0; i < nb; i++) {
      if (status) status[b0 + i] = hst[i];
      if (HMPC_STATUS_CODE(hst[i]) != 0) all_ok = false;
    }
  }
  if (trace) {
    tr[ntr++] = now();
    fprintf(stderr, "[hmpc trace] B=%d us since entry:", B);
    for (int i = 1; i < ntr; i++) fprintf(stderr, " %.0f", tr[i] - tr[0]);
    fprintf(stderr, "  (per chunk: packed, enqueued; then per chunk: synced; end)\n");
  }
  if (!all_ok) { g_err = "hmpc_solve_batch: at least one instance did not reach a KKT point (see status[])"; return HMPC_ERR_NOT_CONVERGED; }
  return HMPC_OK;
}

// ---------------------------------------------------------------------------------------------------
// Part 1: the reference's boundary on a one-robot context (process-global, single caller thread —
// the same contract as the reference's globals, convexMPC_interface.cpp:13-20)
// ---------------------------------------------------------------------------------------------------
namespace {
hmpc_ctx* g_ctx = nullptr;
// the reference's `update` record, the solution buffer and the status word live in ONE page-aligned block that is
// registered with the context, so the one-robot tick runs in place (no packing / staging copies)
struct RefBlock {
  update_data_t update;                       // zero-initialised, like the reference's static `update`
  double soln[12 * HMPC_MAX_HORIZON];
  int status;
};
RefBlock* g_blk = nullptr;
update_data_t g_update_early;  // update_solver_settings may be called before setup_problem
update_data_t& ref_update() { return g_blk ? g_blk->update : g_update_early; }
int g_soln_len = 0;
int g_has_solved = 0;
int g_ref_rc = HMPC_OK;       // result of the last update_problem_data (hmpc_reference_last_rc)
bool g_ref_failing = false;   // inside an episode of failing ticks (the message is printed once per episode)

[[noreturn]] void die(const char* where)
{
  fprintf(stderr, "[hector_mpc_b200] %s: %s\n", where, hmpc_last_error());
  abort();
}
}  // namespace

HMPC_EXTERNC void setup_problem(double dt, int horizon, double mu, double f_max)
{
  if (horizon > 19) {  // SolverMPC.cpp:140-143 throws here; a C boundary must not leak exceptions
    g_err = "horizon is too long!";
    die("setup_problem");
  }
  if (!g_ctx || g_ctx->horizon != horizon) {
    if (g_ctx) hmpc_destroy(g_ctx);
    g_ctx = hmpc_create(1, horizon, 0);  // refuses horizons above HMPC_MAX_HORIZON
    if (!g_ctx) die("setup_problem");
    if (!g_blk) {
      void* mem = nullptr;
      const size_t bytes = (sizeof(RefBlock) + 4095) / 4096 * 4096;
      if (posix_memalign(&mem, 4096, bytes) != 0) { g_err = "out of memory"; die("setup_problem"); }
      memset(mem, 0, bytes);
      g_blk = static_cast<RefBlock*>(mem);
      g_blk->update = g_update_early;
    }
    memset(g_blk->soln, 0, sizeof(g_blk->soln));
    g_soln_len = 12 * horizon;
    // in-place ticks; if registration is not possible the staged path is used (same results)
    if (hmpc_pin_host_buffer(g_ctx, g_blk, (sizeof(RefBlock) + 4095) / 4096 * 4096) != HMPC_OK)
      fprintf(stderr, "[hector_mpc_b200] setup_problem: %s (using staged copies)\n", hmpc_last_error());
  }
  problem_setup s;
  s.dt = (float)dt;
  s.mu = (float)mu;
  s.f_max = (float)f_max;
  s.horizon = horizon;
  hmpc_set_problem(g_ctx, &s);
}

HMPC_EXTERNC void update_problem_data(double* p, double* v, double* q, double* w, double* r, double* joint_angles,
                                      double yaw, double* weights, double* state_trajectory, double* Alpha_K,
                                      int* gait)
{
  if (!g_ctx) { g_err = "update_problem_data called before setup_problem"; die("update_problem_data"); }
  const int N = g_ctx->horizon;
  // double -> float narrowing, convexMPC_interface.cpp:87-99
  for (int i = 0; i < 3; i++) { ref_update().p[i] = (float)p[i]; ref_update().v[i] = (float)v[i]; ref_update().w[i] = (float)w[i]; }
  for (int i = 0; i < 4; i++) ref_update().q[i] = (float)q[i];
  for (int i = 0; i < 6; i++) ref_update().r[i] = (float)r[i];
  for (int i = 0; i < 10; i++) ref_update().joint_angles[i] = (float)joint_angles[i];
  ref_update().yaw = (float)yaw;
  for (int i = 0; i < 12; i++) { ref_update().weights[i] = (float)weights[i]; ref_update().Alpha_K[i] = (float)Alpha_K[i]; }
  for (int i = 0; i < 12 * N; i++) ref_update().traj[i] = (float)state_trajectory[i];
  for (int i = 0; i < 2 * N; i++) ref_update().gait[i] = (unsigned char)gait[i];
  int rc = hmpc_solve_batch(g_ctx, &g_blk->update, 1, g_blk->soln, &g_blk->status);
  g_ref_rc = rc;
  if (rc == HMPC_ERR_NOT_CONVERGED) printf("failed to solve!\n");  // SolverMPC.cpp:714-715 (status word: hmpc_reference_last_status())
  else if (rc != HMPC_OK) {
    // a run-time failure: the controller keeps running on the last wrench and can ask why (hmpc_reference_last_rc)
    const char* ab = getenv("HMPC_REFERENCE_ABORT");
    if (ab && atoi(ab) != 0) die("update_problem_data");
    if (!g_ref_failing)
      fprintf(stderr, "[hector_mpc_b200] update_problem_data: %s — keeping the previous solution (hmpc_reference_last_rc() = %d)\n",
              hmpc_last_error(), rc);
    g_ref_failing = true;
    return;
  }
  g_ref_failing = false;
  g_has_solved = 1;
}

HMPC_EXTERNC double get_solution(int index)
{
  if (!g_has_solved) return 0.f;  // convexMPC_interface.cpp:107
  if (index < 0 || index >= g_soln_len) return 0.0;
  return g_blk->soln[index];
}

HMPC_EXTERNC void update_solver_settings(int max_iter, double rho, double sigma, double solver_alpha, double terminate,
                                         double use_jcqp)
{
  (void)use_jcqp;  // convexMPC_interface.cpp:112-118: stored, not used by the solve
  ref_update().max_iterations = max_iter;
  ref_update().rho = rho;
  ref_update().sigma = sigma;
  ref_update().solver_alpha = solver_alpha;
  ref_update().terminate = terminate;
}

// status word of the last update_problem_data (additive; not part of the reference boundary)
HMPC_EXTERNC int hmpc_reference_last_status(void) { return g_blk ? g_blk->status : 0; }
// result code of the last update_problem_data (additive): see include/hector_mpc_b200.h
HMPC_EXTERNC int hmpc_reference_last_rc(void) { return g_ref_rc; }
