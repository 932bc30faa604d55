// solver.cu — host driver of the device-resident PARSDMM iteration + the C ABI (include/sipb200.h).
//
// Replaces, behind the reference's own call boundary, PARSDMM.jl:25-258, PARSDMM_initialize.jl:6-318,
// argmin_x.jl, cg.jl, rhs_compose.jl, update_y_l.jl, adapt_rho_gamma.jl, stop_PARSDMM.jl, Q_update!.jl.
// The whole iteration runs on the GPU; the host only
//   * launches kernels,
//   * polls a few device scalars (CG / threshold-search "done" flags, the per-iteration log sums),
//   * evaluates the scalar branch logic of stop_PARSDMM.jl / adapt_rho_gamma.jl:55-126 in TF arithmetic.
// There is no CPU compute fallback anywhere in this file.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstring>
#include <array>
#include <limits>
#include <map>
#include <memory>
#include <thread>
#include <unordered_map>
#include <vector>

#include <dlfcn.h>
#include <nccl.h>   // types only: the library is resolved at run time (see NcclApi)

#include "kernels.cuh"
#include <cub/device/device_radix_sort.cuh>   // stable radix sort (library code) for the histogram set only

namespace sipb {

static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }

#define SIPB_REQUIRE(cond, code, msg)   \
  do {                                  \
    if (!(cond)) {                      \
      ::sipb::set_error(msg);           \
      return (code);                    \
    }                                   \
  } while (0)

// NCCL is bound lazily with dlopen/dlsym instead of a link-time dependency: a process that has already
// imported torch keeps using torch's bundled libnccl (same soname), and single-GPU users never load it.
struct NcclApi {
  decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
  decltype(&ncclCommInitRank) CommInitRank = nullptr;
  decltype(&ncclCommDestroy) CommDestroy = nullptr;
  decltype(&ncclAllReduce) AllReduce = nullptr;
  decltype(&ncclAllGather) AllGather = nullptr;
  decltype(&ncclSend) Send = nullptr;
  decltype(&ncclRecv) Recv = nullptr;
  decltype(&ncclGroupStart) GroupStart = nullptr;
  decltype(&ncclGroupEnd) GroupEnd = nullptr;
  decltype(&ncclGetErrorString) GetErrorString = nullptr;
  bool ok = false;
};
static NcclApi* nccl_api() {
  static NcclApi api;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (h) {
#define SIPB_NCCL_SYM(name) api.name = reinterpret_cast<decltype(api.name)>(dlsym(h, "nccl" #name))
      SIPB_NCCL_SYM(GetUniqueId); SIPB_NCCL_SYM(CommInitRank); SIPB_NCCL_SYM(CommDestroy); SIPB_NCCL_SYM(AllReduce);
      SIPB_NCCL_SYM(AllGather); SIPB_NCCL_SYM(Send); SIPB_NCCL_SYM(Recv); SIPB_NCCL_SYM(GroupStart);
      SIPB_NCCL_SYM(GroupEnd); SIPB_NCCL_SYM(GetErrorString);
#undef SIPB_NCCL_SYM
      api.ok = api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.AllReduce && api.AllGather && api.Send &&
               api.Recv && api.GroupStart && api.GroupEnd && api.GetErrorString;
    }
  }
  return &api;
}
#define NCCL(fn) (nccl_api()->fn)

#define SIPB_NCCL_CHECK(expr)                                                              \
  do {                                                                                     \
    ncclResult_t _r = (expr);                                                              \
    if (_r != ncclSuccess) {                                                               \
      ::sipb::set_error(std::string(#expr) + ": " + NCCL(GetErrorString)(_r) + " (" + __FILE__ + \
                        ":" + std::to_string(__LINE__) + ")");                            \
      return SIPB_E_NCCL;                                                                  \
    }                                                                                      \
  } while (0)

// ---------------------------------------------------------------------------------------------
// kernel classes (for the launch counter / CUDA-event table of sipb_log)
// ---------------------------------------------------------------------------------------------
enum KClass {
  KC_SPMV_DOT = 0, KC_CG_INIT, KC_CG_FIN, KC_CG_XR, KC_CG_P, KC_RHS, KC_YL_FUSED, KC_YL_PASS1, KC_YL_PASS2,
  KC_RDUAL, KC_ADAPT, KC_STOP, KC_Q_UPDATE, KC_L1_PASS, KC_RADIX_HIST, KC_TIES, KC_FEAS, KC_VEC_STATS,
  KC_OP_APPLY, KC_PARAMS, KC_FILL, KC_SPMV, KC_COUNT
};
static_assert(KC_COUNT <= SIPB_N_KERNEL_CLASSES, "kernel table too small");
static const char* kClassNames[SIPB_N_KERNEL_CLASSES] = {
    "cds_spmv_dot", "cg_init", "cg_init_fin", "cg_update_xr", "cg_update_p", "rhs_compose", "yl_update_fused",
    "yl_update_pass1", "yl_update_pass2", "r_dual", "adapt_reduce_snapshot", "stop_reduce", "cds_scaled_add",
    "l1_threshold_pass", "topk_radix_hist", "topk_ties", "feasibility", "vec_stats", "op_apply", "proj_params",
    "fill", "cds_spmv", "", ""};

template <typename T>
struct DevBuf {
  T* p = nullptr;       // first owned element (256-byte aligned)
  T* base = nullptr;    // allocation start (p - front)
  size_t n = 0;
  DevBuf() {}
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { release(); }
  void swap(DevBuf& o) {
    std::swap(p, o.p);
    std::swap(base, o.base);
    std::swap(n, o.n);
  }
  void release() {
    if (base) cudaFree(base);
    p = base = nullptr;
    n = 0;
  }
  // `front` / `back` extra elements before / after the owned range (halo planes of a slab)
  cudaError_t alloc(size_t count, size_t front = 0, size_t back = 0) {
    release();
    n = count;
    if (count + front + back == 0) return cudaSuccess;
    const size_t align = 256 / sizeof(T);
    const size_t fpad = (front + align - 1) / align * align;
    cudaError_t e = cudaMalloc(&base, (fpad + count + back) * sizeof(T));
    if (e != cudaSuccess) { base = nullptr; return e; }
    p = base + fpad;
    if (front + back) e = cudaMemset(base, 0, (fpad + count + back) * sizeof(T));
    return e;
  }
};

}  // namespace sipb

using namespace sipb;

// =============================================================================================
// context
// =============================================================================================
struct sipb_ctx {
  int device = 0;
  int num_sms = 148;
  cudaStream_t stream = nullptr;
  cudaStream_t stream_body = nullptr;      // only used while capturing the body of a graph WHILE node
  bool graph_loops = true;                 // device-side CG / l1 loops (SIPB_GRAPH_LOOPS=0: host-driven loops)
  RedScratch rs{nullptr, nullptr};
  RedScratch rs_multi{nullptr, nullptr};   // kYlMulti slices for the multi-set y/l launch
  double* d_scal = nullptr;   // device scalar slots
  double* h_scal = nullptr;   // pinned mirror
  CgState* d_cg = nullptr;
  CgState* h_cg = nullptr;    // pinned
  L1State* d_l1 = nullptr;
  L1State* h_l1 = nullptr;
  SelState* d_sel = nullptr;
  unsigned long long* d_tie_counts = nullptr;
  unsigned long long* d_tie_base = nullptr;   // [kMaxBlocks] exclusive prefix of d_tie_counts (deferred tie handling)
  unsigned int* d_sel_table = nullptr;   // [max_grid()][kSelBins] per-block histograms of the last select level (tie counts)
  bool sel_spec = true;                  // speculative select levels inside pass 1 of the y/l update (SIPB_SEL_SPEC=0: off)
  int l1_skipv = 1;                      // l1 sets: pass 1 skips the store of v while the ball is inactive (SIPB_L1_SKIPV=0: never,
                                         //   2: always — the gated launch then materialises v whenever the ball is active)
  unsigned int* d_counter2 = nullptr;
  int rank = 0, world = 1;
  ncclComm_t comm = nullptr;
  unsigned long long* d_gather = nullptr;   // [world][4] tie counts (all-gather target)
  unsigned long long* d_gather_local = nullptr;   // [4] this rank's tie totals per row block
  // peer-memory path (CUDA IPC over NVLink): mailboxes + counters; see common.cuh
  bool p2p = false;
  PeerMail* d_mail = nullptr;                      // this rank's mailbox (exported)
  void* peer_mail_base[kMaxRanks] = {nullptr};     // imported mappings (to close)
  unsigned long long* d_seq_pv = nullptr;          // [0] seq, [1] pv, [2] bseq
  int* d_p2p_err = nullptr;
  int* h_p2p_err = nullptr;
  CommDev cd_on;                                   // descriptor with the peer path active
  CommDev cd_off;
  PeerBig* d_big = nullptr;                        // this rank's buffer of the small peer all-reduces (exported)
  void* peer_big_base[kMaxRanks] = {nullptr};
  BigDev bd;                                       // valid when p2p
  int64_t peer_collectives = 0;
  // all-reduce of `count` 64-bit words in place: peer memory when the path is up and the payload is small, else NCCL
  template <int OP>
  int small_allreduce(void* d, size_t count, ncclDataType_t dt, ncclRedOp_t op) {
    if (world == 1) return SIPB_OK;
    if (p2p && d_big && count <= (size_t)kBigN) {
      peer_collectives++;
      k_peer_allreduce<OP><<<1, kBigN, 0, stream>>>(bd, reinterpret_cast<unsigned long long*>(d), (int)count);
      return SIPB_OK;
    }
    nccl_calls++;
    SIPB_NCCL_CHECK(NCCL(AllReduce)(d, d, count, dt, op, comm, stream));
    return SIPB_OK;
  }
  std::vector<void*> shared_bufs;                  // exported p vectors: freed at ctx teardown only (see DESIGN)
  // all-gather `bytes` per rank through a device bounce buffer (set-up only)
  int allgather_bytes(const void* mine, void* all, size_t bytes) {
    char* d = nullptr;
    SIPB_CUDA_CHECK(cudaMalloc(&d, bytes * (size_t)(world + 1)));
    SIPB_CUDA_CHECK(cudaMemcpyAsync(d, mine, bytes, cudaMemcpyHostToDevice, stream));
    nccl_calls++;
    SIPB_NCCL_CHECK(NCCL(AllGather)(d, d + bytes, bytes, ncclChar, comm, stream));
    SIPB_CUDA_CHECK(cudaMemcpyAsync(all, d + bytes, bytes * (size_t)world, cudaMemcpyDeviceToHost, stream));
    SIPB_CUDA_CHECK(cudaStreamSynchronize(stream));
    cudaFree(d);
    return SIPB_OK;
  }
  int64_t nccl_calls = 0;
  int64_t l1_graph_runs = 0;
  // sum-all-reduce of `count` doubles in place on the stream (no-op on a single GPU)
  int allreduce(double* d, size_t count) { return small_allreduce<0>(d, count, ncclDouble, ncclSum); }
  int allreduce_u64(unsigned long long* d, size_t count) { return small_allreduce<1>(d, count, ncclUint64, ncclSum); }
  int allreduce_min_u64(unsigned long long* d, size_t count) { return small_allreduce<2>(d, count, ncclUint64, ncclMin); }
  // launch accounting
  bool profile = false;
  int64_t launches[SIPB_N_KERNEL_CLASSES];
  double ms[SIPB_N_KERNEL_CLASSES];
  double bytes[SIPB_N_KERNEL_CLASSES];
  int64_t total_launches = 0;
  struct EvPair { cudaEvent_t a, b; int cls; };
  std::vector<EvPair> ev_used;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev_pool;
  std::vector<std::pair<cudaEvent_t, int>> phase_events;      // (event, phase it closes), reused by every solve
  // algorithmic bytes of the launches of a class: every array the kernel has to read or write counted once
  // (perfect reuse of gathered vectors), the numerator of the roofline in bench.py / DESIGN.md
  void account(int cls, double nbytes) { bytes[cls] += nbytes; }
  void reset_accounting() {
    for (int i = 0; i < SIPB_N_KERNEL_CLASSES; ++i) { launches[i] = 0; ms[i] = 0.0; bytes[i] = 0.0; }
    total_launches = 0;
  }
  int max_grid() const { return std::min(num_sms * 8, kMaxBlocks); }
  int grid_for(i64 work_items) const {
    i64 g = (work_items + kThreads - 1) / kThreads;
    if (g < 1) g = 1;
    return (int)std::min<i64>(g, max_grid());
  }
  // Grid-stride kernels run best with exactly one resident wave: more blocks than fit leave a partial last wave
  // (e.g. 1184 blocks at 5 blocks/SM = 1.6 waves, the second one 60 % full).  The occupancy of each kernel is
  // queried once and cached.
  std::unordered_map<const void*, int> occ_cache;
  int grid_fit(const void* kernel, i64 work_items) {
    auto it = occ_cache.find(kernel);
    int occ;
    if (it == occ_cache.end()) {
      occ = 0;
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, kThreads, 0) != cudaSuccess || occ < 1) {
        cudaGetLastError();
        occ = 4;
      }
      occ_cache[kernel] = occ;
    } else {
      occ = it->second;
    }
    i64 g = (work_items + kThreads - 1) / kThreads;
    if (g < 1) g = 1;
    return (int)std::min<i64>(g, std::min(num_sms * occ, kMaxBlocks));
  }
  void pre_launch(int cls) {
    launches[cls]++;
    total_launches++;
    if (profile) {
      std::pair<cudaEvent_t, cudaEvent_t> pr;
      if (!ev_pool.empty()) { pr = ev_pool.back(); ev_pool.pop_back(); }
      else { cudaEventCreate(&pr.first); cudaEventCreate(&pr.second); }
      cudaEventRecord(pr.first, stream);
      ev_used.push_back({pr.first, pr.second, cls});
    }
  }
  void post_launch() {
    if (profile) cudaEventRecord(ev_used.back().b, stream);
  }
  void collect_profile() {
    if (!profile) return;
    cudaStreamSynchronize(stream);
    for (auto& e : ev_used) {
      float t = 0.f;
      cudaEventElapsedTime(&t, e.a, e.b);
      ms[e.cls] += t;
      ev_pool.push_back({e.a, e.b});
    }
    ev_used.clear();
  }
};

constexpr int kScalSlots = 512;
constexpr int kSlotPerSet = 16;
constexpr int kSlotGlobal = kMaxSets * kSlotPerSet;   // 256

#define LAUNCH(ctx, cls, kern, grid, ...)                         \
  do {                                                            \
    (ctx)->pre_launch(cls);                                       \
    kern<<<(grid), kThreads, 0, (ctx)->stream>>>(__VA_ARGS__);    \
    (ctx)->post_launch();                                         \
  } while (0)
#define LAUNCH1(ctx, cls, kern, ...)                              \
  do {                                                            \
    (ctx)->pre_launch(cls);                                       \
    kern<<<1, 1, 0, (ctx)->stream>>>(__VA_ARGS__);                \
    (ctx)->post_launch();                                         \
  } while (0)

// Copies the scalar slots to the host.  With slabs the slots hold per-rank partial sums: one batched
// Float64 all-reduce makes them global first; the slots are then cleared so that stale entries never
// accumulate across iterations.
static int ctx_sync_scalars(sipb_ctx* c, bool with_loop_state = false) {
  int rc = c->allreduce(c->d_scal, kScalSlots);
  if (rc) return rc;
  SIPB_CUDA_CHECK(cudaMemcpyAsync(c->h_scal, c->d_scal, kScalSlots * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  if (with_loop_state) {     // device-side loops (CG, l1 search): their outcome travels with the scalars
    SIPB_CUDA_CHECK(cudaMemcpyAsync(c->h_cg, c->d_cg, sizeof(CgState), cudaMemcpyDeviceToHost, c->stream));
    SIPB_CUDA_CHECK(cudaMemcpyAsync(c->h_l1, c->d_l1, sizeof(L1State), cudaMemcpyDeviceToHost, c->stream));
    if (c->p2p) SIPB_CUDA_CHECK(cudaMemcpyAsync(c->h_p2p_err, c->d_p2p_err, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  }
  if (c->world > 1) SIPB_CUDA_CHECK(cudaMemsetAsync(c->d_scal, 0, kScalSlots * sizeof(double), c->stream));
  SIPB_CUDA_CHECK(cudaStreamSynchronize(c->stream));
  return SIPB_OK;
}

// =============================================================================================
// small parameter kernels (1 thread)
// =============================================================================================
namespace sipb {

template <typename T>
__global__ void k_l1_begin(const double* stats, double tau, double M, const double* warm, L1State* st,
                           ProjParams<T>* pp, LoopCond lc) {
  loop_set(lc, true);
  const T s1 = (T)stats[0];
  st->tau = tau;
  st->S1 = stats[0];
  st->M = M;
  st->passes = 0;
  if (s1 <= (T)tau) {          // norm(v,1) <= b && return v   (project_l1_Duchi!.jl:23)
    st->done = 1;
    st->theta = -1.0;
    pp->theta = (T)-1;
    loop_set(lc, false);
    return;
  }
  const double w = *warm;
  st->done = 0;
  st->theta = (w > 0.0) ? w : 0.0;
  st->on_left = (w > 0.0) ? 0 : 1;
}
template <typename T>
__global__ void k_l1_end(L1State* st, double* warm, ProjParams<T>* pp) {
  if (st->theta < 0.0) return;   // untouched
  const T th = (T)st->theta;
  pp->theta = th > (T)0 ? th : (T)0;    // theta = max(0, ...)  (project_l1_Duchi!.jl:46)
  *warm = st->theta;
}

// project_l1_Duchi!.jl:42-46: the scan `while u[rho+1] > (sv[rho+1]-b)/(rho+1) && (rho+1) < lv` stops at rho = lv-1,
// so when every entry is active (C == M at the exact root) the reference takes
//   theta = max(0, (sv[lv-1] - b)/(lv-1)),   sv[lv-1] = sum|v| - min|v|
// instead of the exact root (S - b)/M.  `minkey`: min |v| as a magnitude key (k_absmin_key).
template <typename T>
__global__ void k_l1_cap(L1State* st, const unsigned long long* minkey, ProjParams<T>* pp) {
  if (st->theta < 0.0 || st->C != st->M || st->M < 2.0) return;
  T umin;
  if (sizeof(T) == 4) umin = (T)__uint_as_float((unsigned)*minkey);
  else umin = (T)__longlong_as_double((long long)*minkey);
  const T sv = (T)(st->S1 - (double)umin);
  const T th = (sv - (T)st->tau) / (T)(st->M - 1.0);
  pp->theta = th > (T)0 ? th : (T)0;
}

// l2 ball / annulus parameters from sum v^2     (project_l2!.jl:8-13, project_annulus!.jl:8-18)
template <typename T>
__global__ void k_l2_params(const double* stats, int kind, double smin, double smax, double M, ProjParams<T>* pp) {
  const T nl2 = (T)sqrt(stats[1]);
  pp->scale = (T)1;
  pp->fill = (T)NAN;
  if (kind == SIPB_SET_L2) {
    const T sigma = (T)smax;
    if (!(nl2 <= sigma)) pp->scale = sigma / nl2;
  } else {
    const T lo = (T)smin, hi = (T)smax;
    if (lo <= nl2 && nl2 <= hi) return;
    if (nl2 > hi) pp->scale = hi / nl2;
    else if (nl2 < lo && nl2 > (T)0) pp->scale = lo / nl2;
    else if (nl2 < lo && nl2 == (T)0) pp->fill = (T)((double)lo / sqrt(M));
  }
}

// 256 threads.  spec != 0: pass 1 of the y/l update (k_yl_spec) left speculative histograms of the first levels in
// st->spec, built around the guess pp->key_thr (the previous iteration's threshold, still in place): levels are
// consumed for as long as the digits decided so far agree with the guess.
template <typename T>
__global__ void __launch_bounds__(256) k_sel_begin(long long k, long long M, SelState* st, ProjParams<T>* pp, int dbits,
                                                   int spec) {
  __shared__ unsigned long long s_guess;
  if (threadIdx.x == 0) {
    s_guess = pp->key_thr;
    pp->keep_all = (k >= M) ? 1 : 0;
    pp->keep_none = (k <= 0) ? 1 : 0;
    pp->need_ties = 0;
    pp->key_thr = 0ull;
    pp->quota = 0ull;
    pp->count_eq = 0ull;
    st->key_bits = (int)(sizeof(T) * 8);
    st->dbits = dbits;
    st->prefix = 0ull;
    st->k_rem = (unsigned long long)(k > 0 ? k : 0);
    st->count_eq = 0ull;
    st->table_valid = 0;
    st->levels_run = 0;
    st->bits_left = (pp->keep_all || pp->keep_none) ? 0 : st->key_bits;
  }
  for (int b = threadIdx.x; b < kSelBins; b += blockDim.x) st->hist[b] = 0ull;
  __syncthreads();
  if (!spec) return;
  const unsigned long long guess = s_guess;
  constexpr int KB = (int)sizeof(T) * 8;
  // level 0: the threshold lies in the guess's top-digit bucket iff  above < k <= above + |bucket|
  {
    __shared__ unsigned long long s_part[8];
    __shared__ int s_hit;
    unsigned long long mine = 0ull;
    for (int b = threadIdx.x; b < kSelBins; b += blockDim.x) mine += st->spec[b];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
    if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = mine;
    __syncthreads();
    if (threadIdx.x == 0) {
      unsigned long long bucket = 0ull;
      for (int i = 0; i < 8; ++i) bucket += s_part[i];
      const unsigned long long above = st->spec_above, kk = st->k_rem;
      s_hit = 0;
      if (st->bits_left == KB && above < kk && kk <= above + bucket) {
        st->prefix = guess >> (KB - kSpecBits);
        st->k_rem = kk - above;
        st->count_eq = bucket;
        st->bits_left = KB - kSpecBits;
        s_hit = 1;
      }
      st->spec_above = 0ull;
    }
    __syncthreads();
    if (s_hit) {
      for (int lv = 1; lv < kSpecLevels; ++lv) {
        __shared__ int s_go;
        if (threadIdx.x == 0) {
          const int bl = st->bits_left;             // level lv was histogrammed for bl == KB - lv * kSpecBits
          s_go = (bl == KB - lv * kSpecBits) && st->prefix == (guess >> bl);
        }
        __syncthreads();
        if (!s_go) break;                           // block-uniform
        radix_pick_block(st, st->spec + (size_t)(lv - 1) * kSelBins);
      }
    }
  }
  __syncthreads();
  for (int b = threadIdx.x; b < (kSpecLevels - 1) * kSelBins; b += blockDim.x) st->spec[b] = 0ull;
}
// need_ties also when the threshold magnitude is 0 (k > nnz): the surplus zeros then become +0.0, as
// x[sort_ind[k+1:end]] .= 0 writes them (project_cardinality!.jl:19); a -0.0 inside the quota stays -0.0
template <typename T>
__global__ void k_sel_end(SelState* st, ProjParams<T>* pp) {
  if (pp->keep_all || pp->keep_none) return;
  pp->key_thr = st->prefix;
  pp->quota = st->k_rem;
  pp->count_eq = st->count_eq;
  pp->need_ties = (st->count_eq > st->k_rem) ? 1 : 0;
}

// wrappers that read the tie parameters from device memory (no host round trip)
template <typename T>
__global__ void __launch_bounds__(kThreads) k_tie_count_p(i64 M, const T* __restrict__ v, const ProjParams<T>* pp,
                                                          i64 chunk, unsigned long long* counts, const SelState* st,
                                                          const unsigned int* __restrict__ table) {
  if (!pp->need_ties) return;
  const unsigned long long key = pp->key_thr;
  if (st && table && st->table_valid) {
    // the last level of the search ran over the same row partition and kept its per-block histograms: the number of
    // keys equal to the threshold in this block's rows is the entry of the threshold's last digit
    int wl = st->key_bits % st->dbits;
    if (wl == 0) wl = st->dbits;
    if (threadIdx.x == 0)
      counts[blockIdx.x] = (unsigned long long)table[(size_t)blockIdx.x * kSelBins + (unsigned)(key & (unsigned long long)((1 << wl) - 1))];
    return;
  }
  const i64 lo = (i64)blockIdx.x * chunk, hi = min(M, lo + chunk);
  unsigned int c = 0;
  for (i64 r = lo + threadIdx.x; r < hi; r += blockDim.x) c += (mag_key<T>(v[r]) == key) ? 1u : 0u;
  __shared__ unsigned int sm[32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if (lane == 0) sm[w] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long t = 0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += sm[i];
    counts[blockIdx.x] = t;
  }
}
// totals[b] = number of threshold ties in row block b of this rank (slabs)
__global__ void k_tie_totals(const unsigned long long* counts, int nblk, int g, int stride, unsigned long long* totals) {
  // one warp: lanes stride over the per-block counts of each row block
  const int lane = threadIdx.x & 31;
  for (int b = 0; b < 4; ++b) {
    unsigned long long t = 0;
    if (b < nblk)
      for (int i = lane; i < g; i += 32) t += counts[b * stride + i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (lane == 0) totals[b] = t;
  }
}

// Deferred tie handling (single GPU, y/l update): one block of 1024 threads turns the per-chunk tie counts into their
// exclusive prefix `base` (read by pass 2 through ProjDev::tie_base) and settles the one chunk the quota boundary falls
// into in place — every thread walks a contiguous piece of that chunk, the pieces are ranked by a block scan, ties of
// rank >= quota become zero (stable order = index order, project_cardinality!.jl:18-19 with a stable sortperm).
template <typename T>
__global__ void __launch_bounds__(1024) k_tie_cross(i64 M, T* __restrict__ v, const ProjParams<T>* pp, i64 chunk, int g,
                                                    const unsigned long long* __restrict__ counts,
                                                    unsigned long long* __restrict__ base) {
  if (!pp->need_ties) return;
  __shared__ unsigned long long s_warp[32];
  __shared__ unsigned long long s_cross_base;
  __shared__ int s_cross;
  const unsigned long long key = pp->key_thr, quota = pp->quota;
  const int t = threadIdx.x, lane = t & 31, w = t >> 5;
  if (t == 0) s_cross = -1;
  // exclusive prefix of counts[0..g): thread t owns `per` consecutive chunks
  const int per = (g + 1023) / 1024;
  unsigned long long mine = 0ull;
  for (int j = 0; j < per; ++j) {
    const int b = t * per + j;
    if (b < g) mine += counts[b];
  }
  unsigned long long incl = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long up = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += up;
  }
  if (lane == 31) s_warp[w] = incl;
  __syncthreads();
  unsigned long long off = 0ull;
  for (int q = 0; q < w; ++q) off += s_warp[q];
  unsigned long long run = off + incl - mine;
  for (int j = 0; j < per; ++j) {
    const int b = t * per + j;
    if (b < g) {
      const unsigned long long nb = counts[b];
      base[b] = run;
      if (run < quota && run + nb > quota) { s_cross = b; s_cross_base = run; }     // at most one chunk
      run += nb;
    }
  }
  __syncthreads();
  const int cb = s_cross;
  if (cb < 0) return;                                  // the boundary falls between two chunks: nothing to do in place
  const i64 lo = (i64)cb * chunk, hi = min(M, lo + chunk);
  const i64 len = (hi - lo + 1023) / 1024;
  const i64 a0 = min(hi, lo + (i64)t * len), a1 = min(hi, a0 + len);
  unsigned long long c = 0ull;
  for (i64 r = a0; r < a1; ++r) c += (mag_key<T>(v[r]) == key) ? 1ull : 0ull;
  incl = c;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long up = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += up;
  }
  __syncthreads();                                     // s_warp is reused
  if (lane == 31) s_warp[w] = incl;
  __syncthreads();
  off = 0ull;
  for (int q = 0; q < w; ++q) off += s_warp[q];
  unsigned long long rank = s_cross_base + off + incl - c;
  if (rank + c <= quota) return;                       // all ties of this piece are kept
  for (i64 r = a0; r < a1; ++r) {
    if (mag_key<T>(v[r]) == key) {
      if (rank >= quota) v[r] = (T)0;
      ++rank;
    }
  }
}

// `gather` (slabs): all-gathered totals [world][4]; the global index order of the reference's vector is
// row-block major, planes (= ranks) ascending inside a block, so the ties that precede this rank's
// block `blk` are all ties of earlier blocks plus those of lower ranks in the same block.
template <typename T>
__global__ void __launch_bounds__(kThreads) k_tie_zero_p(i64 M, T* __restrict__ v, const ProjParams<T>* pp, i64 chunk,
                                                         const unsigned long long* __restrict__ counts,
                                                         const unsigned long long* __restrict__ gather, int rank,
                                                         int world, int blk) {
  if (!pp->need_ties) return;
  const unsigned long long key = pp->key_thr, quota = pp->quota;
  __shared__ unsigned long long s_part[32];
  __shared__ unsigned int s_warp[32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  // ties that precede this block's rows: the block sums the counts of the lower blocks in parallel (one thread walking
  // ~1000 counters took 0.5 ms on the last blocks)
  unsigned long long b = 0;
  if (threadIdx.x == 0 && gather) {
    for (int bb = 0; bb < blk; ++bb)
      for (int r = 0; r < world; ++r) b += gather[r * 4 + bb];
    for (int r = 0; r < rank; ++r) b += gather[r * 4 + blk];
  }
  for (unsigned i = threadIdx.x; i < blockIdx.x; i += blockDim.x) b += counts[i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) b += __shfl_xor_sync(0xffffffffu, b, o);
  if (lane == 0) s_part[w] = b;
  __syncthreads();
  unsigned long long base = 0ull;
  for (int i = 0; i < nw; ++i) base += s_part[i];
  if (base + counts[blockIdx.x] <= quota) return;
  const i64 lo = (i64)blockIdx.x * chunk, hi = min(M, lo + chunk);
  if (base >= quota) {            // every tie of this block's rows lies beyond the quota: no ranking needed
    for (i64 r = lo + threadIdx.x; r < hi; r += blockDim.x)
      if (mag_key<T>(v[r]) == key) v[r] = (T)0;
    return;
  }
  for (i64 t0 = lo; t0 < hi; t0 += blockDim.x) {
    const i64 r = t0 + threadIdx.x;
    const bool tie = (r < hi) && (mag_key<T>(v[r]) == key);
    const unsigned bal = __ballot_sync(0xffffffffu, tie);
    const unsigned before = __popc(bal & ((1u << lane) - 1u));
    if (lane == 0) s_warp[w] = __popc(bal);
    __syncthreads();
    unsigned wbase = 0, tot = 0;
    for (int i = 0; i < nw; ++i) {
      if (i < w) wbase += s_warp[i];
      tot += s_warp[i];
    }
    if (tie && base + wbase + before >= quota) v[r] = (T)0;
    base += tot;
    __syncthreads();
  }
}

// element-wise projector with parameters read through a device pointer
template <typename T>
struct ProjRef {
  ProjDev<T> P;                 // static part (kind, bounds, vectors, m, rho)
  const ProjParams<T>* dyn;     // dynamic part (may be null for element-wise kinds)
};
template <typename T>
__device__ __forceinline__ ProjDev<T> proj_resolve(const ProjRef<T>& R) {
  ProjDev<T> P = R.P;
  if (R.dyn) {
    P.theta = R.dyn->theta;
    P.scale = R.dyn->scale;
    P.fill = R.dyn->fill;
    P.key_thr = R.dyn->key_thr;
    P.keep_all = R.dyn->keep_all;
    P.keep_none = R.dyn->keep_none;
  }
  return P;
}

// feasibility / in-place projection with dynamic parameters; `ref` (optional) is the vector P(v) is
// compared with (cardinality ties are resolved on a scratch copy)
template <typename T>
__global__ void __launch_bounds__(kThreads) k_feas_dyn(i64 M, T* __restrict__ v, const T* __restrict__ ref,
                                                       const __grid_constant__ ProjDev<T> P0,
                                                       const ProjParams<T>* dyn, int apply, RedScratch rs,
                                                       double* out) {
  ProjDev<T> P = P0;
  if (dyn) {
    P.theta = dyn->theta; P.scale = dyn->scale; P.fill = dyn->fill;
    P.key_thr = dyn->key_thr; P.keep_all = dyn->keep_all; P.keep_none = dyn->keep_none;
  }
  double d[2] = {0.0, 0.0};
  for (i64 r = (i64)blockIdx.x * blockDim.x + threadIdx.x; r < M; r += (i64)gridDim.x * blockDim.x) {
    const T t = v[r];
    const T t0 = ref ? ref[r] : t;
    const T pt = proj_apply<T>(P, t, r);
    const T pf = pt - t0;
    d[0] += (double)pf * (double)pf;
    d[1] += (double)t0 * (double)t0;
    if (apply) v[r] = pt;
  }
  if (grid_sum<2>(d, rs) && threadIdx.x == 0) {
    out[0] = d[0];
    out[1] = d[1];
  }
}

}  // namespace sipb

// =============================================================================================
// operator descriptors (host)
// =============================================================================================
static int64_t op_rows_host(int ndim, const int64_t* n, int op_kind) {
  const int64_t n0 = n[0], n1 = n[1], n2 = (ndim == 3) ? n[2] : 1;
  const int64_t N = n0 * n1 * n2;
  switch (op_kind) {
    case SIPB_OP_IDENTITY: return N;
    case SIPB_OP_DX: return (n0 - 1) * n1 * n2;
    case SIPB_OP_DY: return ndim == 3 ? n0 * (n1 - 1) * n2 : -1;
    case SIPB_OP_DZ: return ndim == 3 ? n0 * n1 * (n2 - 1) : n0 * (n1 - 1);
    case SIPB_OP_TV:
      return ndim == 3 ? (n0 - 1) * n1 * n2 + n0 * (n1 - 1) * n2 + n0 * n1 * (n2 - 1)
                       : (n0 - 1) * n1 + n0 * (n1 - 1);
    case SIPB_OP_DXZ: return ndim == 2 ? (n0 - 1) * (n1 - 1) : -1;
    default: return -1;
  }
}

// Slab geometry of a 3-D problem partitioned along its slowest axis (one process per GPU).
struct SlabGeom {
  bool on = false;
  i64 k0 = 0, k1 = 0;     // owned planes [k0,k1) of the slowest axis
  i64 nlast = 0;          // global extent of the slowest axis
  i64 plane = 0;          // n0*n1
  bool has_lo = false, has_hi = false;
  i64 nloc() const { return k1 - k0; }
  i64 nz_rows() const { return std::min(k1, nlast - 1) - k0; }   // owned row planes of a D_z block
};

// Device copy of an explicit sparse operator (SIPB_OP_SPARSE), both orientations.
template <typename T>
struct SparseDev {
  DevBuf<long long> rp, cp;
  DevBuf<int> ci, ri;
  DevBuf<T> va, vt;
  // validates the host arrays (monotone pointers, indices in range and ascending) and uploads them
  int upload(const sipb_sparse* A, cudaStream_t stream) {
    SIPB_REQUIRE(A && A->rows >= 1 && A->cols >= 1 && A->nnz >= 0, SIPB_E_INVALID, "bad sparse operator");
    SIPB_REQUIRE(A->rowptr && A->colptr && (A->nnz == 0 || (A->colidx && A->rowidx && A->val && A->valt)), SIPB_E_INVALID,
                 "sparse operator with null arrays");
    SIPB_REQUIRE(A->rows < 2147483647ll && A->cols < 2147483647ll, SIPB_E_UNSUPPORTED,
                 "operator with more than 2^31-1 rows or columns per GPU");
    auto check = [](const int64_t* ptr, const int32_t* idx, int64_t nouter, int64_t ninner, int64_t nnz) -> bool {
      if (ptr[0] != 0 || ptr[nouter] != nnz) return false;
      for (int64_t r = 0; r < nouter; ++r) {
        if (ptr[r + 1] < ptr[r]) return false;
        for (int64_t k = ptr[r]; k < ptr[r + 1]; ++k) {
          if (idx[k] < 0 || idx[k] >= ninner) return false;
          if (k > ptr[r] && idx[k] <= idx[k - 1]) return false;
        }
      }
      return true;
    };
    SIPB_REQUIRE(check(A->rowptr, A->colidx, A->rows, A->cols, A->nnz), SIPB_E_INVALID,
                 "CSR arrays of the sparse operator are inconsistent (indices must ascend inside a row)");
    SIPB_REQUIRE(check(A->colptr, A->rowidx, A->cols, A->rows, A->nnz), SIPB_E_INVALID,
                 "CSC arrays of the sparse operator are inconsistent (indices must ascend inside a column)");
    const size_t nz = (size_t)std::max<int64_t>(A->nnz, 1);
    SIPB_CUDA_CHECK(rp.alloc((size_t)A->rows + 1));
    SIPB_CUDA_CHECK(cp.alloc((size_t)A->cols + 1));
    SIPB_CUDA_CHECK(ci.alloc(nz));
    SIPB_CUDA_CHECK(ri.alloc(nz));
    SIPB_CUDA_CHECK(va.alloc(nz));
    SIPB_CUDA_CHECK(vt.alloc(nz));
    static_assert(sizeof(long long) == sizeof(int64_t), "64-bit pointers expected");
    SIPB_CUDA_CHECK(cudaMemcpyAsync(rp.p, A->rowptr, ((size_t)A->rows + 1) * 8, cudaMemcpyHostToDevice, stream));
    SIPB_CUDA_CHECK(cudaMemcpyAsync(cp.p, A->colptr, ((size_t)A->cols + 1) * 8, cudaMemcpyHostToDevice, stream));
    if (A->nnz) {
      SIPB_CUDA_CHECK(cudaMemcpyAsync(ci.p, A->colidx, (size_t)A->nnz * 4, cudaMemcpyHostToDevice, stream));
      SIPB_CUDA_CHECK(cudaMemcpyAsync(ri.p, A->rowidx, (size_t)A->nnz * 4, cudaMemcpyHostToDevice, stream));
      SIPB_CUDA_CHECK(cudaMemcpyAsync(va.p, A->val, (size_t)A->nnz * sizeof(T), cudaMemcpyHostToDevice, stream));
      SIPB_CUDA_CHECK(cudaMemcpyAsync(vt.p, A->valt, (size_t)A->nnz * sizeof(T), cudaMemcpyHostToDevice, stream));
    }
    SIPB_CUDA_CHECK(cudaStreamSynchronize(stream));
    rows = A->rows;
    cols = A->cols;
    return SIPB_OK;
  }
  i64 rows = 0, cols = 0;
  SparseRef<T> ref() const {
    SparseRef<T> r;
    r.rp = rp.p; r.ci = ci.p; r.va = va.p;
    r.cp = cp.p; r.ri = ri.p; r.vt = vt.p;
    r.rows = rows; r.cols = cols;
    return r;
  }
};

// `n` is the GLOBAL grid; with an active slab the descriptor addresses the rank's local planes.
template <typename T>
static int make_op(int ndim, const int64_t* n, const double* h, int op_kind, int block_mode, OpDev* out,
                   const SlabGeom* sg = nullptr) {
  SIPB_REQUIRE(ndim == 2 || ndim == 3, SIPB_E_INVALID, "ndim must be 2 or 3");
  for (int a = 0; a < ndim; ++a)
    SIPB_REQUIRE(n[a] >= 2, SIPB_E_INVALID, "every grid dimension must be at least 2");
  const bool slab = sg && sg->on;
  OpDev op;
  memset(&op, 0, sizeof(op));
  op.kind = op_kind;
  op.mode = block_mode;
  op.n[0] = (unsigned)n[0];
  op.n[1] = (unsigned)n[1];
  op.n[2] = (ndim == 3) ? (unsigned)(slab ? sg->nloc() : n[2]) : 1u;
  op.kofs = slab ? (unsigned)sg->k0 : 0u;
  op.nlast = (ndim == 3) ? (unsigned)n[2] : 1u;
  op.npts = (i64)op.n[0] * op.n[1] * op.n[2];
  op.cols = (block_mode == SIPB_BLOCK_PLAIN) ? op.npts : 2 * op.npts;
  for (int a = 0; a < 3; ++a) {
    // (-1 or 1) ./ h evaluated in TF: get_discrete_Grad.jl:22-23,58-60 with h = TF(comp_grid.d[a])
    const T hh = (a < ndim) ? (T)h[a] : (T)1;
    op.ih[a] = (double)((T)1 / hh);
  }
  op.a_xz = (double)((T)op.ih[1] * (T)op.ih[0]);
  SIPB_REQUIRE(op_rows_host(ndim, n, op_kind) >= 0, SIPB_E_UNSUPPORTED,
               "operator kind not available for this grid dimensionality");
  const int last_axis = ndim - 1;
  auto blk_rows = [&](int a) -> i64 {
    i64 r = 1;
    for (int q = 0; q < 3; ++q) {
      i64 ext = op.n[q];
      if (q == a) ext = (slab && a == 2) ? sg->nz_rows() : ext - 1;
      r *= ext;
    }
    return r;
  };
  switch (op_kind) {
    case SIPB_OP_IDENTITY: op.nblk = 1; break;
    case SIPB_OP_DX: op.nblk = 1; op.axis[0] = 0; break;
    case SIPB_OP_DY: op.nblk = 1; op.axis[0] = 1; break;
    case SIPB_OP_DZ: op.nblk = 1; op.axis[0] = last_axis; break;
    case SIPB_OP_TV:
      op.nblk = ndim;
      for (int b = 0; b < ndim; ++b) op.axis[b] = last_axis - b;   // vcat(D_z[,D_y],D_x)
      break;
    case SIPB_OP_DXZ: op.nblk = 1; break;
    default: SIPB_REQUIRE(false, SIPB_E_UNSUPPORTED, "unknown operator kind");
  }
  op.row_start[0] = 0;
  if (op_kind == SIPB_OP_IDENTITY) op.row_start[1] = op.npts;
  else if (op_kind == SIPB_OP_DXZ) op.row_start[1] = (i64)(op.n[0] - 1) * (op.n[1] - 1);
  else
    for (int b = 0; b < op.nblk; ++b) op.row_start[b + 1] = op.row_start[b] + blk_rows(op.axis[b]);
  op.rows = op.row_start[op.nblk];
  for (int b = op.nblk + 1; b < 4; ++b) op.row_start[b] = op.rows;
  SIPB_REQUIRE(op.rows < (int64_t)2147483647ll && op.cols < (int64_t)2147483647ll, SIPB_E_UNSUPPORTED,
               "operator with more than 2^31-1 rows or columns per GPU");
  for (int b = 0; b < 4; ++b) op.rs[b] = (unsigned)op.row_start[b];
  *out = op;
  return SIPB_OK;
}

// The identity on a vector of M entries: what the fused y/l kernels see for a set with an explicit sparse
// operator, whose s = A x is produced by k_sparse_forward beforehand.
static inline OpDev identity_over(i64 M) {
  OpDev op;
  memset(&op, 0, sizeof(op));
  op.kind = SIPB_OP_IDENTITY;
  op.mode = SIPB_BLOCK_PLAIN;
  op.nblk = 1;
  op.n[0] = (unsigned)M; op.n[1] = 1u; op.n[2] = 1u;
  op.nlast = 1u;
  op.npts = M; op.rows = M; op.cols = M;
  op.row_start[0] = 0;
  for (int b = 1; b < 4; ++b) op.row_start[b] = M;
  for (int b = 0; b < 4; ++b) op.rs[b] = (unsigned)op.row_start[b];
  op.ih[0] = op.ih[1] = op.ih[2] = 1.0;
  return op;
}

static inline bool op_has_slow_axis_block(const OpDev& op) {
  if (op.kind == SIPB_OP_IDENTITY || op.kind == SIPB_OP_DXZ) return false;
  for (int b = 0; b < op.nblk; ++b)
    if (op.axis[b] == 2) return true;
  return false;
}

// Geometry of the tiled SpMV (spmv_tile.cuh) for Q with offsets `offs` on the grid n (slab: nloc local planes
// starting at global plane kofs).  ok = 0 when the matrix / grid is outside what the tiled kernel handles (the
// generic k_spmv then runs): 2-D or Minkowski problems, lines that are not a whole number of 16-byte vectors,
// offsets other than {0, +-1, +-n0, +-n0*n1}, SIPB_SPMV_TILE=0.
template <typename T>
static TileGeom plan_tile(int ndim, const int64_t* n, bool minkowski, const std::vector<int64_t>& offs, i64 nloc,
                          i64 kofs, bool has_lo, bool has_hi, int num_sms) {
  TileGeom g;
  memset(&g, 0, sizeof(g));
  const char* env = getenv("SIPB_SPMV_TILE");
  if (env && env[0] == '0') return g;
  constexpr int VW = Vec<T>::W;
  if (ndim != 3 || minkowski || offs.empty() || (int)offs.size() > kTileDiag) return g;
  const i64 n0 = n[0], n1 = n[1], P = n0 * n1;
  int present = 0;
  if (n0 % VW != 0 || n0 < VW || n1 < 2 || nloc < 1 || P * (nloc + 2) >= ((i64)1 << 31)) return g;
  for (size_t d = 0; d < offs.size(); ++d) {
    const i64 o = offs[d];
    int code = -1;
    if (o == 0) code = 0;
    else if (o == -1) code = 1;
    else if (o == 1) code = 2;
    else if (o == -n0) code = 3;
    else if (o == n0) code = 4;
    else if (o == -P) code = 5;
    else if (o == P) code = 6;
    if (code < 0 || ((present >> code) & 1)) return g;
    g.code[d] = code;
    present |= 1 << code;
    g.dcol[code] = (int)d;
  }
  if (present != (1 << kTileSlots) - 1) return g;    // the full 7-point stencil only
  g.gpl = (int)(n0 / VW);
  if (g.gpl > kThreads) return g;                    // one column group per thread
  g.LPP = kThreads / g.gpl;                          // lines per pass of the CTA
  g.BD = std::min(kThreads, (g.LPP * g.gpl + 31) / 32 * 32);
  // accumulation order: one of the compiled permutations restricted to the slots this matrix has
  g.order = -1;
  for (int ord = 0; ord < kTileNumOrders && g.order < 0; ++ord) {
    size_t d = 0;
    for (int pos = 0; pos < kTileSlots; ++pos)
      if ((present >> tile_order_slot(ord, pos)) & 1) {
        if (d >= offs.size() || g.code[d] != tile_order_slot(ord, pos)) { d = offs.size() + 1; break; }
        ++d;
      }
    if (d == offs.size()) g.order = ord;
  }
  if (g.order < 0) return g;
  const int cap = kTileMinCtas * num_sms;            // resident CTAs
  const size_t smem_budget = (size_t)(226 * 1024) / kTileMinCtas - 3 * 1024;      // per CTA, beside the static part
  const size_t tab_bytes = 27 * kTileDiag * sizeof(T);
  // choose the tile height: few re-read halo lines / planes, all CTA slots busy, at least 3 stages
  double best = 1e300;
  int bestTJ = 0, bestKC = 0, bestNS = 0;
  const int tj_max = (int)std::min<i64>(n1, (i64)g.LPP * TileItems<T>::n);
  for (int tj = 1; tj <= tj_max; ++tj) {
    const int JT = (int)((n1 + tj - 1) / tj);
    const int TJ = (int)((n1 + JT - 1) / JT);
    if (TJ != tj) continue;                          // balanced heights only
    const size_t stage = (size_t)(TJ + 2) * n0 * sizeof(T);
    const int NS = (int)std::min<size_t>(kTileMaxStages, (smem_budget - tab_bytes) / stage);
    if (NS < 3) continue;
    int KC = (int)std::max<i64>(1, std::min<i64>(nloc, cap / JT));
    if (KC > 1 && nloc / KC < 4) KC = (int)std::max<i64>(1, nloc / 4);        // at least ~4 planes per sweep
    const double planes = (double)nloc / KC;
    const double units = (double)JT * KC;
    const double waves = std::ceil(units / cap);
    // time model: a CTA moves (TJ + 2 halo) lines x (planes + 2 extra plane-tiles + ~3 plane-times of pipeline
    // fill); CTAs of one wave run side by side; too few CTAs cannot keep the SMs busy; passes of the CTA that
    // cover no line of the tile idle their threads.  (Measured at 512^3: TJ = 8 / 256 CTAs beats the evenly
    // spread TJ = 7 / 296 CTAs, 326 vs 341 us — taller tiles re-read fewer halo lines.)
    const double passes = std::ceil((double)TJ / g.LPP);
    const double cost = waves * (TJ + 2.0) * (planes + 5.0) * std::max(1.0, 0.5 * cap / units) * (passes * g.LPP / TJ);
    if (cost < best) { best = cost; bestTJ = TJ; bestKC = KC; bestNS = NS; }
  }
  if (!bestTJ) return g;
  g.TJ = bestTJ;
  g.JT = (int)((n1 + g.TJ - 1) / g.TJ);
  g.KC = bestKC;
  g.NS = bestNS;
  g.nloc = (int)nloc;
  g.kofs = (int)kofs;
  g.n2g = (int)n[2];
  g.has_lo = has_lo ? 1 : 0;
  g.has_hi = has_hi ? 1 : 0;
  g.stage_elems = (int)((g.TJ + 2) * n0);
  g.grid = std::min(g.JT * g.KC, cap);
  g.smem_bytes = (size_t)g.NS * g.stage_elems * sizeof(T) + tab_bytes;
  g.ok = 1;
  if (getenv("SIPB_TILE_DEBUG"))
    fprintf(stderr, "[sipb200] tiled SpMV plan: grid %lldx%lldx%lld TJ=%d JT=%d KC=%d NS=%d BD=%d LPP=%d order=%d CTAs=%d smem=%zu\n",
            (long long)n0, (long long)n1, (long long)nloc, g.TJ, g.JT, g.KC, g.NS, g.BD, g.LPP, g.order, g.grid, g.smem_bytes);
  return g;
}
// the tiled kernels use more dynamic shared memory than the default limit: opt in once per instantiation
template <typename K>
static int tile_opt_in(K kernel, size_t bytes) {
  static std::unordered_map<const void*, size_t> done;
  auto it = done.find((const void*)kernel);
  if (it != done.end() && it->second >= bytes) return SIPB_OK;
  SIPB_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(200 * 1024)));
  done[(const void*)kernel] = 200 * 1024;
  return SIPB_OK;
}
// launch k_spmv_tile<T, MODE, ARR, ORD> with the block size / dynamic shared memory of the geometry
template <typename T, int MODE, bool ARR, int ORD>
static int launch_tile_ord(sipb_ctx* c, int cls, const TileGeom& g, const SpmvArgs<T>& a, const TileInit<T>& ti,
                           double* out_dot, const int* done_flag, CgState* st, const CommDev& cd) {
  int rc = tile_opt_in(k_spmv_tile<T, MODE, ARR, ORD>, g.smem_bytes);
  if (rc) return rc;
  c->pre_launch(cls);
  k_spmv_tile<T, MODE, ARR, ORD><<<g.grid, g.BD, g.smem_bytes, c->stream>>>(a, g, ti, c->rs, out_dot, done_flag, st, cd);
  c->post_launch();
  return SIPB_OK;
}
template <typename T, int MODE>
static int launch_tile(sipb_ctx* c, int cls, const TileGeom& g, bool arrays, const SpmvArgs<T>& a, const TileInit<T>& ti,
                       double* out_dot, const int* done_flag, CgState* st, const CommDev& cd) {
  // the array form of the matrix has a tiled body for the plain product only (unit tests, micro-benchmark); the
  // solver streams CDS arrays through the generic kernel, which is at the HBM roofline for them
#define SIPB_TILE_CASE(ORD)                                                                              \
  case ORD:                                                                                              \
    if (arrays) {                                                                                        \
      if constexpr (MODE == 1)                                                                           \
        return launch_tile_ord<T, 1, true, ORD>(c, cls, g, a, ti, out_dot, done_flag, st, cd);           \
      break;                                                                                             \
    }                                                                                                    \
    return launch_tile_ord<T, MODE, false, ORD>(c, cls, g, a, ti, out_dot, done_flag, st, cd);
  switch (g.order) {
    SIPB_TILE_CASE(0)
    SIPB_TILE_CASE(1)
    SIPB_TILE_CASE(2)
    default: break;
  }
#undef SIPB_TILE_CASE
  set_error("tiled SpMV: accumulation order without a compiled body");
  return SIPB_E_STATE;
}
static_assert(kTileNumOrders == 3, "launch_tile dispatches three orders");
// shared-memory opt-in of the class-form kernels of this geometry (outside any stream capture)
template <typename T>
static int tile_prepare(const TileGeom& g) {
  int rc = SIPB_OK;
  switch (g.order) {
    case 0: rc = tile_opt_in(k_spmv_tile<T, 1, false, 0>, g.smem_bytes); if (!rc) rc = tile_opt_in(k_spmv_tile<T, 2, false, 0>, g.smem_bytes); break;
    case 1: rc = tile_opt_in(k_spmv_tile<T, 1, false, 1>, g.smem_bytes); if (!rc) rc = tile_opt_in(k_spmv_tile<T, 2, false, 1>, g.smem_bytes); break;
    case 2: rc = tile_opt_in(k_spmv_tile<T, 1, false, 2>, g.smem_bytes); if (!rc) rc = tile_opt_in(k_spmv_tile<T, 2, false, 2>, g.smem_bytes); break;
    default: break;
  }
  return rc;
}

// A CUDA graph  init -> WHILE(cond) { body } -> tail  built by stream capture: the CG iteration and the l1 threshold
// search loop on the device; the kernel that decides convergence sets the condition (LoopCond, common.cuh).
struct LoopGraph {
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  void destroy() {
    if (exec) cudaGraphExecDestroy(exec);
    if (graph) cudaGraphDestroy(graph);
    exec = nullptr;
    graph = nullptr;
  }
};
// init / body / tail launch kernels on ctx->stream (the body is captured on a second stream that temporarily takes its
// place); each returns a SIPB_* code.
template <typename FInit, typename FBody, typename FTail>
static int build_loop_graph(sipb_ctx* c, LoopGraph& out, FInit init, FBody body, FTail tail) {
  out.destroy();
  cudaStream_t s = c->stream;
  SIPB_CUDA_CHECK(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
  int rc = SIPB_OK;
  cudaGraph_t g = nullptr, done_graph = nullptr;
  auto fail = [&](int code) {
    cudaStreamEndCapture(s, &done_graph);
    if (done_graph) cudaGraphDestroy(done_graph);
    cudaGetLastError();
    return code;
  };
  cudaStreamCaptureStatus st;
  const cudaGraphNode_t* deps = nullptr;
  size_t nd = 0;
  if (cudaStreamGetCaptureInfo(s, &st, nullptr, &g, &deps, &nd) != cudaSuccess || !g) return fail(SIPB_E_CUDA);
  LoopCond lc;
  lc.on = 1;
  if (cudaGraphConditionalHandleCreate(&lc.h, g, 0, cudaGraphCondAssignDefault) != cudaSuccess) return fail(SIPB_E_CUDA);
  if ((rc = init(lc))) return fail(rc);
  if (cudaStreamGetCaptureInfo(s, &st, nullptr, &g, &deps, &nd) != cudaSuccess) return fail(SIPB_E_CUDA);
  cudaGraphNodeParams np = {cudaGraphNodeTypeConditional};
  np.conditional.handle = lc.h;
  np.conditional.type = cudaGraphCondTypeWhile;
  np.conditional.size = 1;
  cudaGraphNode_t cn;
  if (cudaGraphAddNode(&cn, g, deps, nd, &np) != cudaSuccess) return fail(SIPB_E_CUDA);
  cudaGraph_t bg = np.conditional.phGraph_out[0];
  if (cudaStreamUpdateCaptureDependencies(s, &cn, 1, cudaStreamSetCaptureDependencies) != cudaSuccess) return fail(SIPB_E_CUDA);
  // the loop body is captured into the conditional node's own graph on a second stream
  cudaStream_t sb = c->stream_body;
  if (cudaStreamBeginCaptureToGraph(sb, bg, nullptr, nullptr, 0, cudaStreamCaptureModeThreadLocal) != cudaSuccess)
    return fail(SIPB_E_CUDA);
  c->stream = sb;
  rc = body(lc);
  c->stream = s;
  cudaGraph_t bdone = nullptr;
  if (cudaStreamEndCapture(sb, &bdone) != cudaSuccess || rc) return fail(rc ? rc : SIPB_E_CUDA);
  if ((rc = tail())) return fail(rc);
  if (cudaStreamEndCapture(s, &out.graph) != cudaSuccess) { cudaGetLastError(); return SIPB_E_CUDA; }
  if (cudaGraphInstantiate(&out.exec, out.graph, 0) != cudaSuccess) {
    out.destroy();
    cudaGetLastError();
    return SIPB_E_CUDA;
  }
  return SIPB_OK;
}

// =============================================================================================
// problem
// =============================================================================================
struct sipb_problem {
  sipb_ctx* ctx;
  int dtype;
  virtual ~sipb_problem() {}
  virtual int add_set(const sipb_set_desc* d) = 0;
  virtual int set_ata(int idx, const void* R, int64_t rows, const int64_t* offs, int nd) = 0;
  virtual int set_ata_classes(int idx, const void* tab, const int64_t* offs, int nd) = 0;
  virtual int finalize() = 0;
  virtual int solve(const void* m, void* x, void* const* l, void* const* y, const sipb_options* o, sipb_log* log) = 0;
  virtual int q_offsets(std::vector<int64_t>& out) = 0;
  virtual int q_form() const = 0;
  virtual int warm_from(sipb_problem* coarse, const sipb_resample_seg* segs, int nseg) = 0;
};

namespace sipb {

static inline double now_s() {
  return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

template <typename T>
struct SetT {
  sipb_set_desc desc;
  OpDev op;
  i64 M = 0;       // rows held by this rank
  i64 Mglob = 0;   // rows of the global operator
  DevBuf<T> y, l, y_old, s, s0, y0, l0, lhat0;   // s only for reduction-type projectors
  DevBuf<T> lo_vec, hi_vec;
  DevBuf<T> perm;             // SIPB_SET_CARD_SLICE, x / y slices: slice-major scratch copy
  // SIPB_SET_HISTOGRAM: keys / row indices (double buffered) and the scratch space of the radix sort
  DevBuf<typename SortKey<T>::type> hkeys[2];
  DevBuf<unsigned int> hidx[2];
  DevBuf<unsigned char> hsort;
  size_t hsort_bytes = 0;
  int alloc_hist(i64 M_) {
    for (int q = 0; q < 2; ++q) {
      SIPB_CUDA_CHECK(hkeys[q].alloc((size_t)M_));
      SIPB_CUDA_CHECK(hidx[q].alloc((size_t)M_));
    }
    hsort_bytes = 0;
    SIPB_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(nullptr, hsort_bytes, hkeys[0].p, hkeys[1].p, hidx[0].p, hidx[1].p, M_));
    SIPB_CUDA_CHECK(hsort.alloc(hsort_bytes + 256));
    return SIPB_OK;
  }
  SparseDev<T> sparse;        // SIPB_OP_SPARSE: the explicit operator (op is then the identity over the s buffer)
  bool is_sparse = false;
  unsigned td_kofs = 0;       // slabs, fiber modes: global index of the first local plane of the transform-domain grid
  DevBuf<T> ata;              // [nd][ld]   (released once the stencil-class table has been verified)
  DevBuf<T> ata_tab;          // [kMaxClasses][nd] stencil-class form of AtA
  int nd = 0;
  std::vector<int64_t> offs;
  std::vector<int> qcol;      // column of Q for each diagonal of AtA
  bool has_ata = false;
  bool tab_direct = false;    // ata_tab came from the host (sipb_problem_set_ata_classes): nothing to extract / verify
  DevBuf<ProjParams<T>> pp_y, pp_f;   // dynamic projector parameters: y-update / feasibility
  DevBuf<double> warm;        // [2] warm-start thresholds (y-update, feasibility)
  bool z_halo = false;        // slabs: y, l, y_old have a halo plane in front (D_z block)
  int l1_last[2] = {5, 5};    // Newton passes the last l1 threshold search needed (y-update / feasibility)
  bool l1_inactive_prev = false;   // l1 set: the last y-update found sum|v| <= tau (guess for the next pass 1, see skip_v)
  std::map<std::array<const void*, 4>, LoopGraph> l1_graphs;   // device-side search loops, one per (vector, stats, warm, params)
  ~SetT() { for (auto& kv : l1_graphs) kv.second.destroy(); }
};

template <typename T>
struct Problem : sipb_problem {
  int ndim;
  int64_t n[3];
  double h[3];
  bool minkowski, feas_only, finalized = false;
  i64 npts, N;                // grid points, unknowns (2*npts for Minkowski)
  i64 ld;                     // leading dimension of CDS arrays
  std::vector<std::unique_ptr<SetT<T>>> sets;
  std::vector<int64_t> q_offs;
  DevBuf<T> Q, x, x_old, rhs, r, pvec, Ap, m, tmp;
  DevBuf<T> Q_tab;            // [kMaxClasses][nq] stencil-class form of Q (replaces Q when q_classes)
  bool q_classes = false;
  TileGeom tile;              // geometry of the tiled SpMV (tile.ok == 0: generic kernel)
  YlMultiArgs<T> yl_multi;    // argument block of the multi-set y/l launch (rebuilt every iteration)
  i64 maxM = 0;
  bool m_resident = false;
  SlabGeom sg;                // active when the ctx has a communicator with world > 1
  // peer path: p lives in an IPC-exported allocation; the neighbours' p are mapped here
  // peer path: the CG residual r lives in an IPC-exported allocation; the neighbours' r are mapped here (k_cg_p reads
  // their boundary planes to update the local halo planes of p)
  T* r_shared = nullptr;      // owned start of the exported r vector (null => r)
  const T* r_lo = nullptr;    // lower / upper neighbour's r (owned start)
  const T* r_hi = nullptr;
  void* p_lo_base = nullptr;
  void* p_hi_base = nullptr;
  i64 n_lo = 0;
  LoopGraph cg_graph;         // init -> WHILE { SpMV, x/r update, p update } -> zero-fill on rhs == 0
  const void* cg_graph_key[3] = {nullptr, nullptr, nullptr};
  ~Problem() override {
    cg_graph.destroy();
    if (p_lo_base) cudaIpcCloseMemHandle(p_lo_base);
    if (p_hi_base) cudaIpcCloseMemHandle(p_hi_base);
  }
  T* pv() { return pvec.p; }
  T* rv() { return r_shared ? r_shared : r.p; }
  // Export this rank's p vector and import the neighbours' (collective over all ranks).
  int setup_peer_p() {
    sipb_ctx* c = ctx;
    if (!sg.on || !c->p2p) return SIPB_OK;
    const size_t align = 256 / sizeof(T);
    const size_t fpad = ((size_t)sg.plane + align - 1) / align * align;
    void* base = nullptr;
    const size_t bytes = (fpad + (size_t)N + (size_t)sg.plane) * sizeof(T);
    cudaIpcMemHandle_t mine;
    memset(&mine, 0, sizeof(mine));
    int ok = cudaMalloc(&base, bytes) == cudaSuccess && cudaMemset(base, 0, bytes) == cudaSuccess &&
             cudaIpcGetMemHandle(&mine, base) == cudaSuccess;
    cudaGetLastError();
    std::vector<cudaIpcMemHandle_t> all(c->world);
    int rc = c->allgather_bytes(&mine, all.data(), sizeof(mine));
    if (rc) return rc;
    SIPB_REQUIRE(ok, SIPB_E_CUDA, "could not export the r vector for the peer path");
    c->shared_bufs.push_back(base);
    r_shared = reinterpret_cast<T*>(base) + fpad;
    if (sg.has_lo) {
      SIPB_CUDA_CHECK(cudaIpcOpenMemHandle(&p_lo_base, all[c->rank - 1], cudaIpcMemLazyEnablePeerAccess));
      r_lo = reinterpret_cast<const T*>(p_lo_base) + fpad;
      const i64 k0l = n[2] * (c->rank - 1) / c->world, k1l = n[2] * c->rank / c->world;
      n_lo = sg.plane * (k1l - k0l);
    }
    if (sg.has_hi) {
      SIPB_CUDA_CHECK(cudaIpcOpenMemHandle(&p_hi_base, all[c->rank + 1], cudaIpcMemLazyEnablePeerAccess));
      r_hi = reinterpret_cast<const T*>(p_hi_base) + fpad;
    }
    return SIPB_OK;
  }
  i64 Nglob;                  // global number of unknowns (== N on a single GPU)
  int create_error = SIPB_OK;

  Problem(sipb_ctx* c, int dt, int nd_, const int64_t* n_, const double* h_, bool mk, bool fo) {
    ctx = c; dtype = dt; ndim = nd_; minkowski = mk; feas_only = fo;
    memset(&tile, 0, sizeof(tile));
    for (int a = 0; a < 3; ++a) { n[a] = (a < nd_) ? n_[a] : 1; h[a] = (a < nd_) ? h_[a] : 1.0; }
    npts = n[0] * n[1] * n[2];
    Nglob = mk ? 2 * npts : npts;
    if (c->world > 1) {
      // slabs along the slowest axis of a 3-D grid; Minkowski sets couple the halves through the
      // offsets +-N and stay on one GPU (SURVEY 8e)
      if (nd_ != 3 || mk) {
        create_error = SIPB_E_UNSUPPORTED;
      } else {
        sg.on = true;
        sg.nlast = n[2];
        sg.plane = n[0] * n[1];
        sg.k0 = n[2] * c->rank / c->world;
        sg.k1 = n[2] * (c->rank + 1) / c->world;
        sg.has_lo = c->rank > 0;
        sg.has_hi = c->rank < c->world - 1;
        if (sg.nloc() < 1) create_error = SIPB_E_INVALID;
        npts = sg.plane * sg.nloc();
      }
    }
    N = mk ? 2 * npts : npts;
    ld = (N + 63) / 64 * 64;
  }

  ncclDataType_t nccl_type() const { return sizeof(T) == 4 ? ncclFloat : ncclDouble; }

  // Halo exchange of one plane per direction for a vector whose owned part starts at `v` and spans
  // `planes` planes.  up: my last plane -> lower halo (v - plane) of rank+1;
  // down: my first plane -> upper halo (v + planes*plane) of rank-1.  Planes are contiguous: no packing.
  int exchange(T* v, i64 planes, bool up, bool down) {
    if (!sg.on) return SIPB_OK;
    sipb_ctx* c = ctx;
    const size_t cnt = (size_t)sg.plane;
    c->nccl_calls++;
    SIPB_NCCL_CHECK(NCCL(GroupStart)());
    if (up) {
      if (sg.has_hi) SIPB_NCCL_CHECK(NCCL(Send)(v + (planes - 1) * sg.plane, cnt, nccl_type(), c->rank + 1, c->comm, c->stream));
      if (sg.has_lo) SIPB_NCCL_CHECK(NCCL(Recv)(v - sg.plane, cnt, nccl_type(), c->rank - 1, c->comm, c->stream));
    }
    if (down) {
      if (sg.has_lo) SIPB_NCCL_CHECK(NCCL(Send)(v, cnt, nccl_type(), c->rank - 1, c->comm, c->stream));
      if (sg.has_hi) SIPB_NCCL_CHECK(NCCL(Recv)(v + planes * sg.plane, cnt, nccl_type(), c->rank + 1, c->comm, c->stream));
    }
    SIPB_NCCL_CHECK(NCCL(GroupEnd)());
    return SIPB_OK;
  }
  // lower halos of y and l for every set with a D_z block (needed by the rhs / dual-residual gathers);
  // the y_old halo is the previous y halo: it travels with the buffer when y and y_old trade places
  int exchange_yl_halos() {
    if (!sg.on) return SIPB_OK;
    SIPB_NCCL_CHECK(NCCL(GroupStart)());      // one fused NCCL launch for all planes of all sets
    int rc = SIPB_OK;
    for (auto& S : sets) {
      if (!S->z_halo) continue;
      rc = exchange(S->y.p, sg.nz_rows(), true, false);
      if (rc) break;
      rc = exchange(S->l.p, sg.nz_rows(), true, false);
      if (rc) break;
    }
    SIPB_NCCL_CHECK(NCCL(GroupEnd)());
    return rc;
  }

  int add_set(const sipb_set_desc* d) override {
    SIPB_REQUIRE(!finalized, SIPB_E_STATE, "problem already finalized");
    SIPB_REQUIRE((int)sets.size() < kMaxSets, SIPB_E_UNSUPPORTED, "too many sets");
    SIPB_REQUIRE(d->set_kind >= SIPB_SET_BOUNDS_SCALAR && d->set_kind <= SIPB_SET_KIND_MAX, SIPB_E_UNSUPPORTED,
                 "set type is outside the device hot path (rank, nuclear and subspace sets are rejected)");
    const bool fiber = d->set_kind == SIPB_SET_BOUNDS_FIBER || d->set_kind == SIPB_SET_CARD_FIBER ||
                       d->set_kind == SIPB_SET_CARD_SLICE;
    if (fiber) {
      SIPB_REQUIRE(!minkowski, SIPB_E_UNSUPPORTED, "fiber modes are not available for Minkowski problems");
      SIPB_REQUIRE(d->fiber_axis >= 0 && d->fiber_axis < ndim, SIPB_E_INVALID, "fiber axis outside the grid");
      // slabs cut the slowest axis: everything that stays inside a plane works rank-locally — per-fiber bounds along
      // any axis (element-wise; the bound of a z fiber is indexed by the GLOBAL plane), per-fiber cardinality along x / y,
      // per-slice cardinality of z slices (= planes).  Fibers / slices that cross slabs would need a distributed select.
      if (sg.on) {
        SIPB_REQUIRE(!(d->set_kind == SIPB_SET_CARD_FIBER && d->fiber_axis == 2), SIPB_E_UNSUPPORTED,
                     "per-fiber cardinality along the slab axis is single-GPU (the fibers cross the slabs)");
        SIPB_REQUIRE(!(d->set_kind == SIPB_SET_CARD_SLICE && d->fiber_axis != 2), SIPB_E_UNSUPPORTED,
                     "per-slice cardinality of x / y slices is single-GPU (the slices cross the slabs)");
      }
      SIPB_REQUIRE(d->op_kind != SIPB_OP_TV, SIPB_E_INVALID,
                   "fiber modes need a single-block operator (the TV output is not a grid)");
    }
    SIPB_REQUIRE(minkowski ? d->block_mode != SIPB_BLOCK_PLAIN : d->block_mode == SIPB_BLOCK_PLAIN, SIPB_E_INVALID,
                 "block_mode inconsistent with the Minkowski flag of the problem");
    if (d->set_kind == SIPB_SET_L1) SIPB_REQUIRE(d->max > 0.0, SIPB_E_INVALID, "Radius of L1 ball is negative");
    if (d->set_kind == SIPB_SET_HISTOGRAM)
      SIPB_REQUIRE(!sg.on, SIPB_E_UNSUPPORTED, "the histogram set (a global sort) is single-GPU");
    auto S = std::make_unique<SetT<T>>();
    S->desc = *d;
    S->desc.sparse = nullptr;        // the host arrays are not kept
    int rc;
    if (d->op_kind == SIPB_OP_SPARSE) {
      // custom_TD_OP (setup_constraints.jl:70-72): an explicit sparse matrix with N columns
      SIPB_REQUIRE(!sg.on && !minkowski && !fiber, SIPB_E_UNSUPPORTED,
                   "explicit sparse operators are single-GPU, non-Minkowski, matrix/tensor mode");
      SIPB_REQUIRE(d->sparse && d->sparse->cols == npts, SIPB_E_INVALID, "sparse operator must have prod(n) columns");
      rc = S->sparse.upload(d->sparse, ctx->stream);
      if (rc) return rc;
      S->is_sparse = true;
      S->op = identity_over(d->sparse->rows);
      S->M = S->op.rows;
      S->Mglob = S->M;
    } else {
      rc = make_op<T>(ndim, n, h, d->op_kind, d->block_mode, &S->op, &sg);
      if (rc) return rc;
      S->M = S->op.rows;
      S->Mglob = op_rows_host(ndim, n, d->op_kind);
    }
    S->z_halo = sg.on && op_has_slow_axis_block(S->op);
    cudaError_t e = cudaSuccess;
    auto A = [&](DevBuf<T>& b) { if (e == cudaSuccess) e = b.alloc((size_t)S->M); };
    // slabs: y, l, y_old of a set with a D_z block carry the neighbour's last row plane in front
    auto AH = [&](DevBuf<T>& b) { if (e == cudaSuccess) e = b.alloc((size_t)S->M, S->z_halo ? (size_t)sg.plane : 0, 0); };
    AH(S->y); AH(S->l); AH(S->y_old); A(S->s0); A(S->y0); A(S->l0); A(S->lhat0);
    if (!proj_is_elementwise(d->set_kind) || S->is_sparse) A(S->s);
    if (d->set_kind == SIPB_SET_CARD_SLICE && d->fiber_axis != 2) A(S->perm);
    if (e == cudaSuccess) e = S->pp_y.alloc(1);
    if (e == cudaSuccess) e = S->pp_f.alloc(1);
    if (e == cudaSuccess) e = S->warm.alloc(2);
    SIPB_CUDA_CHECK(e);
    SIPB_CUDA_CHECK(cudaMemsetAsync(S->warm.p, 0, 2 * sizeof(double), ctx->stream));
    SIPB_CUDA_CHECK(cudaMemsetAsync(S->pp_y.p, 0, sizeof(ProjParams<T>), ctx->stream));
    SIPB_CUDA_CHECK(cudaMemsetAsync(S->pp_f.p, 0, sizeof(ProjParams<T>), ctx->stream));
    if (fiber) {
      SIPB_REQUIRE(d->td_n[0] * d->td_n[1] * d->td_n[2] == S->Mglob && d->td_n[0] >= 1 && d->td_n[1] >= 1 && d->td_n[2] >= 1,
                   SIPB_E_INVALID, "td_n does not match the rows of the operator");
      if (sg.on) {     // the rank-local transform-domain grid: this rank's planes of the (single) row block
        SIPB_REQUIRE(S->M % (d->td_n[0] * d->td_n[1]) == 0, SIPB_E_INVALID, "slab rows are not whole planes of td_n");
        S->desc.td_n[2] = S->M / (d->td_n[0] * d->td_n[1]);
        S->td_kofs = (unsigned)sg.k0;
      }
    }
    if (d->set_kind == SIPB_SET_HISTOGRAM) { rc = S->alloc_hist(S->M); if (rc) return rc; }
    if (d->set_kind == SIPB_SET_BOUNDS_VECTOR || d->set_kind == SIPB_SET_BOUNDS_FIBER || d->set_kind == SIPB_SET_HISTOGRAM) {
      SIPB_REQUIRE(d->min_vec && d->max_vec, SIPB_E_INVALID, "vector bounds need min_vec and max_vec");
      const size_t nb = d->set_kind == SIPB_SET_BOUNDS_FIBER ? (size_t)d->td_n[d->fiber_axis] : (size_t)S->M;
      SIPB_CUDA_CHECK(S->lo_vec.alloc(nb));
      SIPB_CUDA_CHECK(S->hi_vec.alloc(nb));
      SIPB_CUDA_CHECK(cudaMemcpyAsync(S->lo_vec.p, d->min_vec, nb * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
      SIPB_CUDA_CHECK(cudaMemcpyAsync(S->hi_vec.p, d->max_vec, nb * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
      SIPB_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
      S->desc.min_vec = S->desc.max_vec = nullptr;
    }
    maxM = std::max<i64>(maxM, S->M);
    sets.push_back(std::move(S));
    return SIPB_OK;
  }

  int set_ata(int idx, const void* R, int64_t rows, const int64_t* offs, int nd) override {
    SIPB_REQUIRE(!finalized, SIPB_E_STATE, "problem already finalized");
    SIPB_REQUIRE(idx >= 0 && idx < (int)sets.size(), SIPB_E_INVALID, "set index out of range");
    SIPB_REQUIRE(rows == N, SIPB_E_INVALID, "AtA must have N rows");
    SIPB_REQUIRE(nd >= 1 && nd <= kMaxDiag, SIPB_E_UNSUPPORTED, "number of diagonals outside [1,32]");
    SetT<T>& S = *sets[idx];
    SIPB_CUDA_CHECK(S.ata.alloc((size_t)ld * nd));
    SIPB_CUDA_CHECK(cudaMemsetAsync(S.ata.p, 0, (size_t)ld * nd * sizeof(T), ctx->stream));
    SIPB_CUDA_CHECK(cudaMemcpy2DAsync(S.ata.p, ld * sizeof(T), R, N * sizeof(T), N * sizeof(T), nd,
                                      cudaMemcpyHostToDevice, ctx->stream));
    SIPB_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    S.nd = nd;
    S.offs.assign(offs, offs + nd);
    S.has_ata = true;
    return SIPB_OK;
  }

  int set_ata_classes(int idx, const void* tab, const int64_t* offs, int nd) override {
    SIPB_REQUIRE(!finalized, SIPB_E_STATE, "problem already finalized");
    SIPB_REQUIRE(idx >= 0 && idx < (int)sets.size(), SIPB_E_INVALID, "set index out of range");
    SIPB_REQUIRE(nd >= 1 && nd <= kMaxDiag, SIPB_E_UNSUPPORTED, "number of diagonals outside [1,32]");
    SIPB_REQUIRE(n[0] * n[1] * n[2] < ((i64)1 << 31) && !(minkowski && sg.on), SIPB_E_UNSUPPORTED,
                 "stencil-class tables need fewer than 2^31 grid points");
    SetT<T>& S = *sets[idx];
    SIPB_REQUIRE(!S.is_sparse, SIPB_E_INVALID, "custom sparse operators come as CDS arrays (sipb_problem_set_ata)");
    SIPB_CUDA_CHECK(S.ata_tab.alloc((size_t)kMaxClasses * nd));
    SIPB_CUDA_CHECK(cudaMemcpyAsync(S.ata_tab.p, tab, (size_t)kMaxClasses * nd * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
    SIPB_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    S.nd = nd;
    S.offs.assign(offs, offs + nd);
    S.has_ata = true;
    S.tab_direct = true;
    return SIPB_OK;
  }

  int finalize() override {
    SIPB_REQUIRE(!finalized, SIPB_E_STATE, "problem already finalized");
    SIPB_REQUIRE(!sets.empty(), SIPB_E_INVALID, "no sets");
    for (auto& S : sets) SIPB_REQUIRE(S->has_ata, SIPB_E_STATE, "AtA missing for a set");
    if (!feas_only)
      SIPB_REQUIRE(sets.back()->desc.set_kind == SIPB_SET_DISTANCE, SIPB_E_INVALID,
                   "the last set must be the distance term unless feasibility_only");
    for (size_t i = 0; i + 1 < sets.size(); ++i)
      SIPB_REQUIRE(sets[i]->desc.set_kind != SIPB_SET_DISTANCE, SIPB_E_INVALID, "distance term must be last");
    // Q_offsets = unique(all_offsets) over the zero-padded 999x99 table, column-major
    // (PARSDMM_initialize.jl:217-221): offsets of AtA[1], then 0, then the unseen ones of AtA[2], ...
    q_offs.clear();
    auto push_unique = [&](int64_t o) {
      if (std::find(q_offs.begin(), q_offs.end(), o) == q_offs.end()) q_offs.push_back(o);
    };
    SIPB_REQUIRE(sets.size() <= 99, SIPB_E_UNSUPPORTED, "more than 99 operators");
    for (size_t i = 0; i < sets.size(); ++i) {
      for (int64_t o : sets[i]->offs) push_unique(o);
      push_unique(0);   // padding zeros of column i (every column is padded: nd <= 32 < 999)
    }
    SIPB_REQUIRE((int)q_offs.size() <= kMaxDiag, SIPB_E_UNSUPPORTED, "Q has more than 32 diagonals");
    for (auto& S : sets) {
      S->qcol.resize(S->nd);
      for (int k = 0; k < S->nd; ++k) {
        auto it = std::find(q_offs.begin(), q_offs.end(), S->offs[k]);
        SIPB_REQUIRE(it != q_offs.end(), SIPB_E_MISSING_DIAG, "diagonal missing in Q");
        S->qcol[k] = (int)(it - q_offs.begin());
      }
    }
    { int rc = detect_classes(); if (rc) return rc; }
    cudaError_t e = cudaSuccess;
    auto A = [&](DevBuf<T>& b, size_t cnt) { if (e == cudaSuccess) e = b.alloc(cnt); };
    if (q_classes) A(Q_tab, (size_t)kMaxClasses * q_offs.size());
    else A(Q, (size_t)ld * q_offs.size());
    const size_t halo = sg.on ? (size_t)sg.plane : 0;      // one plane on each side (max |offset| of Q)
    auto AH = [&](DevBuf<T>& b, size_t cnt) { if (e == cudaSuccess) e = b.alloc(cnt, halo, halo); };
    AH(x, (size_t)N); A(x_old, (size_t)N); A(rhs, (size_t)N); A(r, (size_t)N); AH(pvec, (size_t)N);
    A(Ap, (size_t)N); AH(m, (size_t)N); A(tmp, (size_t)std::max<i64>(maxM, N));
    SIPB_CUDA_CHECK(e);
    if (sg.on)
      for (int64_t o : q_offs)
        SIPB_REQUIRE(std::llabs((long long)o) <= sg.plane, SIPB_E_UNSUPPORTED, "CDS offset wider than one halo plane");
    { int rc = setup_peer_p(); if (rc) return rc; }
    tile = plan_tile<T>(ndim, n, minkowski, q_offs, sg.on ? sg.nloc() : n[2], sg.on ? sg.k0 : 0, sg.on && sg.has_lo,
                        sg.on && sg.has_hi, ctx->num_sms);
    if (tile.ok && q_classes) { int rc = tile_prepare<T>(tile); if (rc) return rc; }
    finalized = true;
    return SIPB_OK;
  }

  ClassGeom class_geom() const {
    ClassGeom g;
    g.n[0] = (unsigned)n[0]; g.n[1] = (unsigned)n[1]; g.n[2] = (unsigned)n[2];
    g.npts = (unsigned)(n[0] * n[1] * n[2]);     // GLOBAL grid points (rows per Minkowski half)
    g.nhalf = minkowski ? 2 : 1;
    g.kofs = sg.on ? (unsigned)sg.k0 : 0u;
    g.nz_loc = sg.on ? (unsigned)sg.nloc() : (unsigned)n[2];
    return g;
  }
  // Do all AtA_i have one value per stencil class and diagonal (kernels.cuh, "Stencil classes")?  Then keep
  // the class tables only: Q becomes a [classes][nq] table and the SpMV stops streaming matrix entries.
  // SIPB_Q_CLASSES=0 keeps the array form (A/B measurements, tests of the general path).
  int detect_classes() {
    q_classes = false;
    const char* env = getenv("SIPB_Q_CLASSES");
    int ok = !(env && env[0] == '0');
    if (n[0] * n[1] * n[2] >= ((i64)1 << 31)) ok = 0;
    if (minkowski && sg.on) ok = 0;
    sipb_ctx* c = ctx;
    bool any_direct = false, all_direct = true;
    for (auto& S : sets) { any_direct = any_direct || S->tab_direct; all_direct = all_direct && S->tab_direct; }
    if (any_direct) {
      // class tables handed over by the host: there is no array to fall back to
      SIPB_REQUIRE(ok, SIPB_E_STATE, "stencil-class tables were passed although SIPB_Q_CLASSES=0 asks for CDS arrays");
      SIPB_REQUIRE(all_direct, SIPB_E_STATE,
                   "either every AtA comes as a stencil-class table or every AtA comes as a CDS array");
      q_classes = true;
      return SIPB_OK;
    }
    if (ok) {
      int* d_bad = (int*)c->d_counter2;
      SIPB_CUDA_CHECK(cudaMemsetAsync(d_bad, 0, sizeof(int), c->stream));
      const ClassGeom g = class_geom();
      const i64 row0 = sg.on ? sg.plane * sg.k0 : 0;
      for (auto& S : sets) {
        SIPB_CUDA_CHECK(S->ata_tab.alloc((size_t)kMaxClasses * S->nd));
        const int cnt = kMaxClasses * S->nd;
        LAUNCH(c, KC_Q_UPDATE, k_class_extract<T>, (cnt + kThreads - 1) / kThreads, (const T*)S->ata.p, ld, S->nd, g,
               S->ata_tab.p);
        LAUNCH(c, KC_Q_UPDATE, k_class_verify<T>, c->grid_for(N), (const T*)S->ata.p, ld, S->nd, N, row0, g,
               (const T*)S->ata_tab.p, d_bad);
      }
      int bad = 0;
      SIPB_CUDA_CHECK(cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
      SIPB_CUDA_CHECK(cudaStreamSynchronize(c->stream));
      SIPB_CUDA_CHECK(cudaMemsetAsync(d_bad, 0, sizeof(int), c->stream));
      ok = bad ? 0 : 1;
    }
    if (c->world > 1) {        // every rank must take the same path (the SpMV kernels differ)
      double v = ok ? 0.0 : 1.0;
      SIPB_CUDA_CHECK(cudaMemcpyAsync(c->d_scal, &v, sizeof(double), cudaMemcpyHostToDevice, c->stream));
      int rc = c->allreduce(c->d_scal, 1);
      if (rc) return rc;
      SIPB_CUDA_CHECK(cudaMemcpyAsync(&v, c->d_scal, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
      SIPB_CUDA_CHECK(cudaStreamSynchronize(c->stream));
      SIPB_CUDA_CHECK(cudaMemsetAsync(c->d_scal, 0, sizeof(double), c->stream));
      ok = v == 0.0;
    }
    if (ok) {
      for (auto& S : sets) S->ata.release();
      q_classes = true;
    } else {
      for (auto& S : sets) S->ata_tab.release();
    }
    return SIPB_OK;
  }
  // Q (+)= alpha * AtA_i in whichever form the problem holds       (CDS_scaled_add!.jl:16-22)
  void q_add(SetT<T>& S, T alpha) {
    sipb_ctx* c = ctx;
    if (q_classes) {
      QCols qc;
      for (int k = 0; k < S.nd; ++k) qc.c[k] = S.qcol[k];
      const int cnt = kMaxClasses * S.nd;
      LAUNCH(c, KC_Q_UPDATE, k_class_axpy<T>, (cnt + kThreads - 1) / kThreads, Q_tab.p, (int)q_offs.size(),
             (const T*)S.ata_tab.p, S.nd, qc, alpha);
    } else {
      const int gN = c->grid_for((N + Vec<T>::W - 1) / Vec<T>::W);
      for (int k = 0; k < S.nd; ++k)
        LAUNCH(c, KC_Q_UPDATE, k_cds_axpy<T>, gN, N, Q.p + (size_t)S.qcol[k] * ld, (const T*)(S.ata.p + (size_t)k * ld),
               alpha);
    }
  }

  int q_form() const override { return q_classes ? 1 : 0; }
  int q_offsets(std::vector<int64_t>& out) override {
    SIPB_REQUIRE(finalized, SIPB_E_STATE, "problem not finalized");
    out = q_offs;
    return SIPB_OK;
  }

  // Row blocks of a vector in the global (row-block major) order on slabs: first global row, rows per z plane,
  // and whether the block differences along z (a D_z block has one row plane fewer than the grid).
  struct SlabBlock { i64 start, plane; bool dz; };
  std::vector<SlabBlock> slab_blocks(int vec) const {
    std::vector<SlabBlock> out;
    if (vec < 0 || sets[vec]->op.kind == SIPB_OP_IDENTITY) {
      out.push_back({0, n[0] * n[1], false});
      return out;
    }
    const OpDev& op = sets[vec]->op;
    i64 start = 0;
    for (int b = 0; b < op.nblk; ++b) {
      const int a = op.axis[b];
      const SlabBlock k{start, (n[0] - (a == 0)) * (n[1] - (a == 1)), a == 2};
      out.push_back(k);
      start += k.plane * (n[2] - k.dz);
    }
    return out;
  }
  // planes [k0, k1) of block `k` stored by `rank` (the rule of SlabGeom::nz_rows)
  std::pair<i64, i64> slab_planes(const SlabBlock& k, int rank) const {
    const i64 nz = n[2], k0 = nz * rank / ctx->world, k1 = nz * (rank + 1) / ctx->world;
    return {k0, k.dz ? std::min(k1, nz - 1) : k1};
  }
  // Collective: every rank's rows of the slab vector `local` (vector id `vec`: -1 = x, else a set's l / y) land at
  // their global positions in `glob`, so each rank holds the whole vector in the reference's order.
  int gather_global(int vec, const T* local, T* glob) {
    sipb_ctx* c = ctx;
    const auto blks = slab_blocks(vec);
    i64 loc = 0;
    for (const auto& k : blks) {          // own rows: a device copy
      const auto pl = slab_planes(k, c->rank);
      const i64 cnt = k.plane * (pl.second - pl.first);
      if (cnt > 0)
        SIPB_CUDA_CHECK(cudaMemcpyAsync(glob + k.start + k.plane * pl.first, local + loc, cnt * sizeof(T),
                                        cudaMemcpyDeviceToDevice, c->stream));
      loc += cnt;
    }
    c->nccl_calls++;
    SIPB_NCCL_CHECK(NCCL(GroupStart)());
    loc = 0;
    for (const auto& k : blks) {
      const auto mine = slab_planes(k, c->rank);
      const i64 cnt = k.plane * (mine.second - mine.first);
      for (int r = 0; r < c->world; ++r) {
        if (r == c->rank) continue;
        const auto pl = slab_planes(k, r);
        const i64 rcnt = k.plane * (pl.second - pl.first);
        if (cnt > 0) SIPB_NCCL_CHECK(NCCL(Send)(local + loc, (size_t)cnt, nccl_type(), r, c->comm, c->stream));
        if (rcnt > 0)
          SIPB_NCCL_CHECK(NCCL(Recv)(glob + k.start + k.plane * pl.first, (size_t)rcnt, nccl_type(), r, c->comm, c->stream));
      }
      loc += cnt;
    }
    SIPB_NCCL_CHECK(NCCL(GroupEnd)());
    return SIPB_OK;
  }

  // device-side nearest-neighbour warm start from a coarser problem (PARSDMM_multi_level.jl:61-82).  On slabs the
  // segments address global vectors: each coarse vector is gathered whole on every rank, and every rank resamples the
  // rows it stores of each fine vector.
  int warm_from(sipb_problem* coarse_, const sipb_resample_seg* segs, int nseg) override {
    SIPB_REQUIRE(finalized && coarse_ && segs, SIPB_E_STATE, "warm_from needs two finalized problems");
    SIPB_REQUIRE(coarse_->dtype == dtype && coarse_->ctx == ctx, SIPB_E_INVALID, "problems differ in dtype / context");
    Problem<T>* co = static_cast<Problem<T>*>(coarse_);
    SIPB_REQUIRE(co->finalized && co->sets.size() == sets.size(), SIPB_E_INVALID, "level problems have different sets");
    SIPB_REQUIRE(co->sg.on == sg.on, SIPB_E_INVALID, "one level problem is slab-decomposed, the other is not");
    sipb_ctx* c = ctx;
    const int p = (int)sets.size();
    // validate every segment before the first collective, so that all ranks fail alike
    for (int q = 0; q < nseg; ++q) {
      const sipb_resample_seg& g = segs[q];
      i64 ns = 1, nd = 1;
      for (int a = 0; a < 3; ++a) {
        SIPB_REQUIRE(g.src_shape[a] >= 1 && g.dst_shape[a] >= 1, SIPB_E_INVALID, "bad resampling shape");
        ns *= g.src_shape[a];
        nd *= g.dst_shape[a];
      }
      SIPB_REQUIRE(g.vec >= -1 && g.vec < p, SIPB_E_INVALID, "set index out of range");
      const i64 src_len = g.vec < 0 ? (sg.on ? co->Nglob : co->N) : (sg.on ? co->sets[g.vec]->Mglob : co->sets[g.vec]->M);
      const i64 dst_len = g.vec < 0 ? (sg.on ? Nglob : N) : (sg.on ? sets[g.vec]->Mglob : sets[g.vec]->M);
      SIPB_REQUIRE(g.src_off >= 0 && g.src_off + ns <= src_len && g.dst_off >= 0 && g.dst_off + nd <= dst_len,
                   SIPB_E_INVALID, "resampling segment outside its vector");
    }
    DevBuf<T> stage;       // slabs: one whole coarse vector at a time
    if (sg.on) {
      i64 big = co->Nglob;
      for (auto& S : co->sets) big = std::max<i64>(big, S->Mglob);
      SIPB_CUDA_CHECK(stage.alloc((size_t)big));
    }
    // source vectors in the order x, l_0, y_0, l_1, y_1, ...
    for (int v = -1; v < 2 * p; ++v) {
      const int vec = v < 0 ? -1 : v / 2;
      T* dst_vec = vec < 0 ? x.p : (v % 2 ? sets[vec]->y.p : sets[vec]->l.p);
      const T* src_vec = vec < 0 ? co->x.p : (v % 2 ? co->sets[vec]->y.p : co->sets[vec]->l.p);
      bool used = false;
      for (int q = 0; q < nseg; ++q) used = used || segs[q].vec == vec;
      if (!used) continue;        // every rank passes the same segments, so all ranks skip the same gathers
      if (sg.on) {
        int rc = co->gather_global(vec, src_vec, stage.p);
        if (rc) return rc;
        src_vec = stage.p;
      }
      for (int q = 0; q < nseg; ++q) {
        const sipb_resample_seg& g = segs[q];
        if (g.vec != vec) continue;
        const i64 nd = g.dst_shape[0] * g.dst_shape[1] * g.dst_shape[2];
        auto launch = [&](T* dst, i64 q0, i64 q1) {
          LAUNCH(c, KC_OP_APPLY, k_resample_nn<T>, c->grid_for(q1 - q0), src_vec + g.src_off, dst, g.src_shape[0],
                 g.src_shape[1], g.src_shape[2], g.dst_shape[0], g.dst_shape[1], g.dst_shape[2], q0, q1);
        };
        if (!sg.on) {
          launch(dst_vec + g.dst_off, 0, nd);
          continue;
        }
        // this rank's rows of each destination block: one global range per block, stored contiguously
        i64 loc = 0;
        for (const auto& k : slab_blocks(vec)) {
          const auto pl = slab_planes(k, c->rank);
          const i64 gs = k.start + k.plane * pl.first, ge = k.start + k.plane * pl.second;
          const i64 a = std::max(gs, (i64)g.dst_off), b = std::min(ge, (i64)g.dst_off + nd);
          if (a < b) launch(dst_vec + loc + (a - gs), a - g.dst_off, b - g.dst_off);
          loc += ge - gs;
        }
      }
    }
    SIPB_CUDA_CHECK(cudaGetLastError());
    SIPB_CUDA_CHECK(cudaStreamSynchronize(c->stream));
    return SIPB_OK;
  }

  // ---- helpers ------------------------------------------------------------------------------
  SpmvArgs<T> spmv_args(const T* xin, T* yout) const {
    SpmvArgs<T> a;
    a.R = Q.p; a.ld = ld; a.nd = (int)q_offs.size();
    a.tab = q_classes ? Q_tab.p : nullptr;
    a.gn[0] = (unsigned)n[0]; a.gn[1] = (unsigned)n[1]; a.gn[2] = (unsigned)n[2];
    a.npts = (unsigned)(n[0] * n[1] * n[2]);
    for (int j = 0; j < a.nd; ++j) a.off[j] = q_offs[j];
    // constants of the class-form fast path
    a.fast = 0; a.amask = 0u; a.maxoff = 0;
    for (int j = 0; j < 8; ++j) a.off32[j] = 0;
    for (int q = 0; q < 2; ++q) {
      const unsigned d = (unsigned)n[q];
      int l = 0;
      while ((1ull << l) < d) ++l;
      a.div_m[q] = (unsigned)(((1ull << (31 + l)) + d - 1) / d);
      a.div_s[q] = 31 + l;
    }
    if (q_classes && a.nd <= kFastDiag) {
      a.fast = 1;
      for (int j = 0; j < a.nd; ++j) {
        const i64 o = q_offs[j];
        a.maxoff = std::max<i64>(a.maxoff, o < 0 ? -o : o);
        a.off32[j] = (int)o;
        if (o % Vec<T>::W == 0) a.amask |= 1u << j;
      }
      if (a.maxoff >= ((i64)1 << 30)) a.fast = 0;
    }
    a.N = N; a.row0 = sg.on ? sg.plane * sg.k0 : 0; a.Nglob = Nglob; a.x = xin; a.y = yout;
    a.x_lo = nullptr; a.x_hi = nullptr; a.n_lo = 0;
    return a;
  }
  // SpMV on p with the neighbours' planes read through peer pointers
  SpmvArgs<T> spmv_args_peer(T* yout) {
    // the halo planes of p are local on every path: NCCL fills them, or k_cg_p computes them from the neighbours' r
    return spmv_args(pv(), yout);
  }

  ProjDev<T> proj_static(const SetT<T>& S, T rho_dist) const {
    ProjDev<T> P;
    memset(&P, 0, sizeof(P));
    P.kind = S.desc.set_kind;
    P.lo = (T)S.desc.min;
    P.hi = (T)S.desc.max;
    P.lo_vec = S.lo_vec.p;
    P.hi_vec = S.hi_vec.p;
    P.m = m.p;
    for (int a = 0; a < 3; ++a) P.td[a] = (unsigned)std::max<int64_t>(S.desc.td_n[a], 1);
    P.fiber_axis = S.desc.fiber_axis;
    P.td_kofs = S.td_kofs;
    P.rho = (S.desc.set_kind == SIPB_SET_PROX_L1) ? (T)S.desc.max : rho_dist;
    P.theta = (T)-1; P.scale = (T)1; P.fill = (T)NAN; P.key_thr = 0ull; P.keep_all = 1; P.keep_none = 0;
    return P;
  }

  // per-fiber cardinality in place (project_cardinality!.jl:23-113)
  void card_fiber(SetT<T>& S, T* v) {
    sipb_ctx* c = ctx;
    const sipb_set_desc& d = S.desc;
    const unsigned d0 = (unsigned)d.td_n[0], d1 = (unsigned)d.td_n[1], d2 = (unsigned)d.td_n[2];
    if (d.set_kind == SIPB_SET_CARD_SLICE) {
      // every slice orthogonal to fiber_axis is one long "fiber" once it is contiguous (project_cardinality!.jl:115-146)
      const i64 M = (i64)d0 * d1 * d2;
      if (d.fiber_axis == 2) {                        // z: the n3 planes are contiguous already
        LAUNCH(c, KC_TIES, k_card_fiber_contig<T>, c->grid_for((i64)d2 * 32), v, (i64)d2, d0 * d1, (long long)d.k);
        return;
      }
      const i64 nsl = d.fiber_axis == 0 ? d0 : d1;
      const unsigned L = d.fiber_axis == 0 ? d1 * d2 : d0 * d2;
      LAUNCH(c, KC_TIES, k_slice_permute<T>, c->grid_for(M), (const T*)v, S.perm.p, d0, d1, d2, d.fiber_axis, 0);
      LAUNCH(c, KC_TIES, k_card_fiber_contig<T>, c->grid_for(nsl * 32), S.perm.p, nsl, L, (long long)d.k);
      LAUNCH(c, KC_TIES, k_slice_permute<T>, c->grid_for(M), (const T*)S.perm.p, v, d0, d1, d2, d.fiber_axis, 1);
      return;
    }
    if (d.fiber_axis == 0) {
      const i64 nfib = (i64)d1 * d2;
      LAUNCH(c, KC_TIES, k_card_fiber_contig<T>, c->grid_for(nfib * 32), v, nfib, d0, (long long)d.k);
    } else {
      const i64 nfib = d.fiber_axis == 1 ? (i64)d0 * d2 : (i64)d0 * d1;
      LAUNCH(c, KC_TIES, k_card_fiber_strided<T>, c->grid_for(nfib), v, d0, d1, d2, d.fiber_axis, (long long)d.k);
    }
  }

  // Computes the dynamic parameters of a reduction-type projector for the vector `v` whose stats
  // (sum|v|, sum v^2, nnz) sit in d_scal[stat_slot..].  No host synchronisation except the polling
  // of the l1 Newton iteration.
  // tie_defer (single GPU, cardinality): instead of zeroing the surplus ties in place, leave the per-chunk prefix in
  // d_tie_base for the consumer (pass 2 of the y/l update) and return the chunk length through *tie_defer
  int projector_params(SetT<T>& S, T* v, int stat_slot, ProjParams<T>* pp, double* warm, bool allow_tie_zero,
                       bool spec = false, i64* tie_defer = nullptr) {
    sipb_ctx* c = ctx;
    const int kind = S.desc.set_kind;
    const i64 M = S.M;               // rank-local rows
    const i64 Mg = S.Mglob;          // rows of the global operator
    const int fused = sg.on ? 0 : 1; // single GPU: the reducing kernel also performs the scalar step
    double* stats = c->d_scal + stat_slot;
    int rc = c->allreduce(stats, 3);
    if (rc) return rc;
    if (kind == SIPB_SET_L1) {
      const bool peer = sg.on && c->p2p;
      const int g_l1 = c->grid_fit((const void*)k_l1_pass<T>, (M + Vec<T>::W - 1) / Vec<T>::W);
      unsigned long long* mk = c->d_tie_counts;
      if (c->graph_loops && !c->profile && (!sg.on || (peer && c->d_big))) {
        // the whole search as one graph launch: begin -> WHILE { pass [, step] } -> end -> lv-1 cap (device-side
        // decisions only; on slabs the pass publishes its partial (C, S) to the peers' mailboxes, k_l1_step collects
        // them and decides, and the cap's minimum is a small peer all-reduce every rank takes part in)
        LoopGraph& lg = S.l1_graphs[{(const void*)v, (const void*)stats, (const void*)warm, (const void*)pp}];
        if (!lg.exec) {
          rc = build_loop_graph(
              c, lg,
              [&](const LoopCond& lc) {
                LAUNCH1(c, KC_PARAMS, k_l1_begin<T>, stats, (double)(T)S.desc.max, (double)Mg, warm, c->d_l1, pp, lc);
                return SIPB_OK;
              },
              [&](const LoopCond& lc) {
                if (fused) {
                  LAUNCH(c, KC_L1_PASS, k_l1_pass<T>, g_l1, M, (const T*)v, c->rs, c->d_l1, 1, c->cd_off, lc);
                } else {
                  const LoopCond off{0, 0};
                  LAUNCH(c, KC_L1_PASS, k_l1_pass<T>, g_l1, M, (const T*)v, c->rs, c->d_l1, 0, c->cd_on, off);
                  LAUNCH1(c, KC_PARAMS, k_l1_step, c->d_l1, c->cd_on, lc);
                }
                return SIPB_OK;
              },
              [&]() {
                LAUNCH1(c, KC_PARAMS, k_l1_end<T>, c->d_l1, warm, pp);
                if (cudaMemsetAsync(mk, 0xff, sizeof(unsigned long long), c->stream) != cudaSuccess) return SIPB_E_CUDA;
                LAUNCH(c, KC_L1_PASS, k_absmin_key<T>, c->grid_for(M), M, (const T*)v, mk, (const L1State*)c->d_l1);
                if (sg.on) { int r2 = c->allreduce_min_u64(mk, 1); if (r2) return r2; }
                LAUNCH1(c, KC_PARAMS, k_l1_cap<T>, c->d_l1, (const unsigned long long*)mk, pp);
                return SIPB_OK;
              });
          if (rc) { set_error("could not build the l1 search graph"); return rc; }
        }
        SIPB_CUDA_CHECK(cudaGraphLaunch(lg.exec, c->stream));
        c->total_launches += 1;
        c->l1_graph_runs += 1;
      } else {
        const LoopCond off{0, 0};
        LAUNCH1(c, KC_PARAMS, k_l1_begin<T>, stats, (double)(T)S.desc.max, (double)Mg, warm, c->d_l1, pp, off);
        int launched = 0;
        int& last = S.l1_last[warm == S.warm.p ? 0 : 1];
        for (;;) {
          // passes are queued speculatively (they return at once after `done`); the warm-started search mostly
          // repeats the pass count of the previous iteration, so the first batch is sized from it
          const int batch = (launched == 0) ? std::min(std::max(last + 1, 2), 6) : 8;
          for (int b = 0; b < batch; ++b) {
            LAUNCH(c, KC_L1_PASS, k_l1_pass<T>, g_l1, M, v, c->rs, c->d_l1, fused, peer ? c->cd_on : c->cd_off, off);
            if (!fused) {
              if (!peer && (rc = c->allreduce(&c->d_l1->C, 2))) return rc;
              LAUNCH1(c, KC_PARAMS, k_l1_step, c->d_l1, peer ? c->cd_on : c->cd_off, off);
            }
          }
          launched += batch;
          SIPB_CUDA_CHECK(cudaMemcpyAsync(c->h_l1, c->d_l1, sizeof(L1State), cudaMemcpyDeviceToHost, c->stream));
          SIPB_CUDA_CHECK(cudaStreamSynchronize(c->stream));
          if (c->h_l1->done || launched >= 256) break;
        }
        SIPB_REQUIRE(c->h_l1->done && !c->h_l1->failed, SIPB_E_STATE, "l1 threshold search did not converge");
        last = c->h_l1->passes;
        LAUNCH1(c, KC_PARAMS, k_l1_end<T>, c->d_l1, warm, pp);
        if (c->h_l1->theta >= 0.0 && c->h_l1->C == c->h_l1->M && Mg >= 2) {
          // every entry is above the threshold: reproduce the reference's lv-1 cap (project_l1_Duchi!.jl:42-46)
          SIPB_CUDA_CHECK(cudaMemsetAsync(mk, 0xff, sizeof(unsigned long long), c->stream));
          LAUNCH(c, KC_L1_PASS, k_absmin_key<T>, c->grid_for(M), M, (const T*)v, mk, (const L1State*)nullptr);
          if (sg.on && (rc = c->allreduce_min_u64(mk, 1))) return rc;
          LAUNCH1(c, KC_PARAMS, k_l1_cap<T>, c->d_l1, (const unsigned long long*)mk, pp);
        }
      }
    } else if (kind == SIPB_SET_HISTOGRAM) {
      // sortperm + clamp by the sorted bounds + inverse permutation, in place; the apply pass is a pass-through
      LAUNCH(c, KC_TIES, k_hist_keys<T>, c->grid_for(M), M, (const T*)v, S.hkeys[0].p, S.hidx[0].p);
      size_t tb = S.hsort_bytes;
      SIPB_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(S.hsort.p, tb, S.hkeys[0].p, S.hkeys[1].p, S.hidx[0].p, S.hidx[1].p, M, 0,
                                                      (int)(8 * sizeof(typename SortKey<T>::type)), c->stream));
      LAUNCH(c, KC_TIES, k_hist_apply<T>, c->grid_for(M), M, v, (const unsigned int*)S.hidx[1].p, (const T*)S.lo_vec.p,
             (const T*)S.hi_vec.p);
    } else if (kind == SIPB_SET_CARD_FIBER || kind == SIPB_SET_CARD_SLICE) {
      card_fiber(S, v);            // projects every fiber in place; the apply pass is then a pass-through
    } else if (kind == SIPB_SET_L2 || kind == SIPB_SET_ANNULUS) {
      LAUNCH1(c, KC_PARAMS, k_l2_params<T>, stats, kind, S.desc.min, S.desc.max, (double)Mg, pp);
    } else if (kind == SIPB_SET_CARDINALITY) {
      // single GPU: 11-bit digits (3 levels for Float32), every level over the row partition of the tie kernels, the last
      // one keeping its per-block histograms; `spec`: pass 1 of the y/l update already histogrammed the first levels
      // around the previous threshold (k_yl_spec).  Slabs: 8-bit digits, one small all-reduce per level.
      const int dbits = sg.on ? 8 : kSpecBits;
      const int nlev = ((int)sizeof(T) * 8 + dbits - 1) / dbits;
      const int g_sel = c->max_grid();
      const i64 chunk_sel = ((M + g_sel - 1) / g_sel + kThreads - 1) / kThreads * kThreads;
      c->pre_launch(KC_PARAMS);
      k_sel_begin<T><<<1, 256, 0, c->stream>>>((long long)S.desc.k, (long long)Mg, c->d_sel, pp, dbits, spec ? 1 : 0);
      c->post_launch();
      for (int q = 0; q < nlev; ++q) {                // (a level decided by the speculation returns at once)
        if (fused) {
          LAUNCH(c, KC_RADIX_HIST, k_radix_hist<T>, g_sel, M, v, c->d_sel, c->d_counter2, 1, chunk_sel, c->d_sel_table);
        } else {
          LAUNCH(c, KC_RADIX_HIST, k_radix_hist<T>, c->grid_for(M), M, v, c->d_sel, c->d_counter2, 0, (i64)0,
                 (unsigned int*)nullptr);
          rc = c->allreduce_u64(c->d_sel->hist, 256);
          if (rc) return rc;
          c->pre_launch(KC_PARAMS);
          k_radix_pick<<<1, 256, 0, c->stream>>>(c->d_sel);
          c->post_launch();
        }
      }
      LAUNCH1(c, KC_PARAMS, k_sel_end<T>, c->d_sel, pp);
      if (allow_tie_zero) {
        if (!sg.on) {
          const int g = c->max_grid();
          const i64 chunk = ((M + g - 1) / g + kThreads - 1) / kThreads * kThreads;
          LAUNCH(c, KC_TIES, k_tie_count_p<T>, g, M, v, pp, chunk, c->d_tie_counts, (const SelState*)c->d_sel,
                 (const unsigned int*)c->d_sel_table);
          if (tie_defer) {
            // pass 2 of the y/l update zeroes the ties of the chunks beyond the quota boundary (ProjDev::tie_base);
            // only the chunk the boundary falls into is settled here
            c->pre_launch(KC_TIES);
            k_tie_cross<T><<<1, 1024, 0, c->stream>>>(M, v, pp, chunk, g, c->d_tie_counts, c->d_tie_base);
            c->post_launch();
            *tie_defer = chunk;
          } else {
            LAUNCH(c, KC_TIES, k_tie_zero_p<T>, g, M, v, pp, chunk, c->d_tie_counts, (const unsigned long long*)nullptr,
                   0, 1, 0);
          }
        } else {
          // index-ordered ties across slabs: per row block tie totals are all-gathered (4 x world counters)
          const int nb = S.op.kind == SIPB_OP_IDENTITY ? 1 : S.op.nblk;
          const int g = std::min(c->max_grid(), kMaxBlocks / nb);       // the count table holds kMaxBlocks entries
          for (int b = 0; b < nb; ++b) {
            const i64 Mb = S.op.row_start[b + 1] - S.op.row_start[b];
            const i64 chunk = ((std::max<i64>(Mb, 1) + g - 1) / g + kThreads - 1) / kThreads * kThreads;
            LAUNCH(c, KC_TIES, k_tie_count_p<T>, g, Mb, v + S.op.row_start[b], pp, chunk, c->d_tie_counts + (size_t)b * g,
                   (const SelState*)nullptr, (const unsigned int*)nullptr);
          }
          // all-gather of the 4 per-block totals == sum-all-reduce of a [world][4] table in which a rank fills its row
          SIPB_CUDA_CHECK(cudaMemsetAsync(c->d_gather, 0, sizeof(unsigned long long) * 4 * c->world, c->stream));
          c->pre_launch(KC_TIES);
          k_tie_totals<<<1, 32, 0, c->stream>>>(c->d_tie_counts, nb, g, g, c->d_gather + 4 * c->rank);
          c->post_launch();
          rc = c->allreduce_u64(c->d_gather, (size_t)4 * c->world);
          if (rc) return rc;
          for (int b = 0; b < nb; ++b) {
            const i64 Mb = S.op.row_start[b + 1] - S.op.row_start[b];
            const i64 chunk = ((std::max<i64>(Mb, 1) + g - 1) / g + kThreads - 1) / kThreads * kThreads;
            LAUNCH(c, KC_TIES, k_tie_zero_p<T>, g, Mb, v + S.op.row_start[b], pp, chunk, c->d_tie_counts + (size_t)b * g,
                   (const unsigned long long*)c->d_gather, c->rank, c->world, b);
          }
        }
      }
    }
    return SIPB_OK;
  }

  // relative feasibility numerator/denominator of the vector sv (= A x) -> d_scal[slot], [slot+1]
  // in_loop: the feasibility logged every 10th iteration (update_y_l.jl:90-94) relies on P_sub mutating its
  // argument; the reference's slice-mode cardinality does NOT for x / y slices (project_cardinality!.jl:115-118:
  // permutedims copies), so there the logged value is ||s - s|| / ||s|| = 0 — reproduced here.
  int feasibility_of(SetT<T>& S, T* sv, int slot, bool in_loop = false) {
    sipb_ctx* c = ctx;
    const i64 M = S.M;
    ProjDev<T> P = proj_static(S, (T)0);
    if (in_loop && S.desc.set_kind == SIPB_SET_CARD_SLICE && S.desc.fiber_axis != 2) {
      LAUNCH(c, KC_FEAS, k_feas_dyn<T>, c->grid_for(M), M, sv, (const T*)sv, P, (const ProjParams<T>*)S.pp_f.p, 0, c->rs,
             c->d_scal + slot);
      return SIPB_OK;
    }
    if (proj_is_elementwise(S.desc.set_kind)) {
      LAUNCH(c, KC_FEAS, k_feas_dyn<T>, c->grid_for(M), M, sv, (const T*)nullptr, P, (const ProjParams<T>*)nullptr, 0,
             c->rs, c->d_scal + slot);
      return SIPB_OK;
    }
    const int stat_slot = slot + 10;
    LAUNCH(c, KC_VEC_STATS, k_vec_stats<T>, c->grid_for(M), M, sv, c->rs, c->d_scal + stat_slot);
    T* vec = sv;
    const T* ref = nullptr;
    if (S.desc.set_kind == SIPB_SET_CARDINALITY || S.desc.set_kind == SIPB_SET_CARD_FIBER ||
        S.desc.set_kind == SIPB_SET_CARD_SLICE || S.desc.set_kind == SIPB_SET_HISTOGRAM) {   // in-place work on a scratch copy
      SIPB_CUDA_CHECK(cudaMemcpyAsync(tmp.p, sv, M * sizeof(T), cudaMemcpyDeviceToDevice, c->stream));
      vec = tmp.p;
      ref = sv;
    }
    int rc = projector_params(S, vec, stat_slot, S.pp_f.p, S.warm.p + 1, true);
    if (rc) return rc;
    LAUNCH(c, KC_FEAS, k_feas_dyn<T>, c->grid_for(M), M, vec, ref, P, (const ProjParams<T>*)S.pp_f.p, 0, c->rs,
           c->d_scal + slot);
    return SIPB_OK;
  }

  // device CG on Q (cg.jl:44-128).  parsdmm_it > 0 selects the argmin_x tolerance rule.
  // Slabs: the halos of `xv` must be valid on entry; they are valid again on exit.  Every rank launches
  // the same sequence (the control scalars are all-reduced, hence identical), so the NCCL calls match.
  int run_cg(const T* b, T* xv, T* x_old_out, int parsdmm_it, double tol, int max_iter, int predicted,
             int* iters, double* relres, int* flag, bool* deferred = nullptr) {
    sipb_ctx* c = ctx;
    CgState* h = c->h_cg;
    int rc;
    // only the control fields are (re)written; tol_prev persists on the device between calls
    h->maxit = max_iter;
    h->parsdmm_it = parsdmm_it;
    h->tol = tol;
    SIPB_CUDA_CHECK(cudaMemcpyAsync(&c->d_cg->maxit, &h->maxit, sizeof(int), cudaMemcpyHostToDevice, c->stream));
    SIPB_CUDA_CHECK(cudaMemcpyAsync(&c->d_cg->parsdmm_it, &h->parsdmm_it, sizeof(int), cudaMemcpyHostToDevice, c->stream));
    if (parsdmm_it == 0)
      SIPB_CUDA_CHECK(cudaMemcpyAsync(&c->d_cg->tol, &h->tol, sizeof(double), cudaMemcpyHostToDevice, c->stream));
    const bool peer = r_shared != nullptr;            // peer-memory collectives instead of NCCL inside the CG
    T* rr = rv();
    const CommDev& cd = peer ? c->cd_on : c->cd_off;
    T* pp = pv();
    const i64 nvecN = (N + Vec<T>::W - 1) / Vec<T>::W;
    // (k_cg_init measured faster with two waves than with one: 2.03 vs 2.68 ms per solve at 200^3)
    const int g_init = c->grid_for(nvecN), g_mv = c->grid_fit((const void*)k_spmv<T, true>, nvecN),
              g_xr = c->grid_fit((const void*)k_cg_xr<T>, nvecN), g_p = c->grid_fit((const void*)k_cg_p<T>, nvecN);
    const bool tiled = tile.ok && q_classes;
    // r = b - Qx, p = r, x_old = x, tolerance rule / early exits        (argmin_x.jl:33-37, cg.jl:47-76)
    auto launch_init = [&](const LoopCond& lc) -> int {
      if (tiled) {
        const TileInit<T> ti{b, rr, pp, x_old_out};
        if ((rc = launch_tile<T, 2>(c, KC_CG_INIT, tile, false, spmv_args(xv, nullptr), ti, nullptr, nullptr, c->d_cg, cd)))
          return rc;
      } else {
        LAUNCH(c, KC_CG_INIT, k_cg_init<T>, g_init, spmv_args(xv, nullptr), b, rr, pp, x_old_out, c->rs, c->d_cg, cd);
      }
      if (!peer && (rc = c->allreduce(&c->d_cg->bb, 2))) return rc;          // bb, rr are adjacent
      LAUNCH1(c, KC_CG_FIN, k_cg_init_fin<T>, c->d_cg, cd, lc);
      if (peer)      // p = r on the halo planes: the neighbours' boundary planes of r (complete: their partials were collected)
        LAUNCH(c, KC_CG_INIT, k_p_halo_init<T>, c->grid_for(sg.plane), N, sg.plane, pp, r_lo, r_hi, n_lo);
      return SIPB_OK;
    };
    // one CG iteration                                                  (cg.jl:84-114)
    auto launch_iter = [&](const LoopCond& lc, const int* done_flag) -> int {
      if (!peer && (rc = exchange(pp, sg.nloc(), true, true))) return rc;     // halo planes of p
      if (tiled) {
        const TileInit<T> ti{nullptr, nullptr, nullptr, nullptr};
        if ((rc = launch_tile<T, 1>(c, KC_SPMV_DOT, tile, false, spmv_args_peer(Ap.p), ti, &c->d_cg->pAp, done_flag, c->d_cg, cd)))
          return rc;
      } else {
        LAUNCH(c, KC_SPMV_DOT, (k_spmv<T, true>), g_mv, spmv_args_peer(Ap.p), c->rs, &c->d_cg->pAp, done_flag, cd);
      }
      if (!peer && (rc = c->allreduce(&c->d_cg->pAp, 1))) return rc;      // peer path: collected inside k_cg_xr
      LAUNCH(c, KC_CG_XR, k_cg_xr<T>, g_xr, N, xv, rr, pp, Ap.p, c->rs, c->d_cg, cd, sg.on ? sg.plane : (i64)0);
      if (!peer && (rc = c->allreduce(&c->d_cg->rr_new, 1))) return rc;   // peer path: collected inside k_cg_p
      LAUNCH(c, KC_CG_P, k_cg_p<T>, g_p, N, (const T*)rr, pp, c->rs, c->d_cg, cd, sg.on ? sg.plane : (i64)0, lc,
             peer ? r_lo : (const T*)nullptr, peer ? r_hi : (const T*)nullptr, n_lo);
      return SIPB_OK;
    };
    const double vecN = (double)N * sizeof(T);
    const double q_rows = q_classes ? 0.0 : (double)q_offs.size();       // matrix words streamed per row
    c->account(KC_CG_INIT, (q_rows + 4 + (x_old_out ? 1 : 0)) * vecN);   // Q, x, b -> r, p (, x_old)
    if (deferred) {
      // Device-side loop: ONE graph launch runs the prologue, iterates until the convergence test of cg.jl:103 (or
      // maxIter, or alpha < 0) ends the WHILE node, and zero-fills x for a zero right-hand side.  The host does not
      // wait: iteration count, relres and flag are read with the per-iteration scalars (finish_cg).
      if (!cg_graph.exec || cg_graph_key[0] != (const void*)b || cg_graph_key[1] != (const void*)xv ||
          cg_graph_key[2] != (const void*)x_old_out) {
        rc = build_loop_graph(
            c, cg_graph, [&](const LoopCond& lc) { return launch_init(lc); },
            [&](const LoopCond& lc) { return launch_iter(lc, (const int*)nullptr); },
            [&]() {
              LAUNCH(c, KC_FILL, k_cg_zero_x<T>, c->grid_for(N), N, xv, (const CgState*)c->d_cg);
              return SIPB_OK;
            });
        if (rc) { set_error("could not build the CG loop graph"); return rc; }
        cg_graph_key[0] = b; cg_graph_key[1] = xv; cg_graph_key[2] = x_old_out;
      }
      SIPB_CUDA_CHECK(cudaGraphLaunch(cg_graph.exec, c->stream));
      c->total_launches += 1;
      if ((rc = exchange(xv, sg.nloc(), true, true))) return rc;            // halo planes of the new x
      *deferred = true;
      return SIPB_OK;
    }
    const LoopCond off{0, 0};
    if ((rc = launch_init(off))) return rc;
    int launched = 0;
    int batch = std::max(1, predicted);
    for (;;) {
      for (int q = 0; q < batch && launched < max_iter; ++q, ++launched)
        if ((rc = launch_iter(off, (const int*)&c->d_cg->done))) return rc;
      SIPB_CUDA_CHECK(cudaMemcpyAsync(h, c->d_cg, sizeof(CgState), cudaMemcpyDeviceToHost, c->stream));
      if (peer) SIPB_CUDA_CHECK(cudaMemcpyAsync(c->h_p2p_err, c->d_p2p_err, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
      SIPB_CUDA_CHECK(cudaStreamSynchronize(c->stream));
      if (peer) SIPB_REQUIRE(*c->h_p2p_err == 0, SIPB_E_NCCL, "peer-memory collective timed out (a rank stopped participating)");
      if (h->done || launched >= max_iter) break;
      batch = std::max(2, launched / 2);
    }
    account_cg_loops(h);
    if (h->flag == -9) SIPB_CUDA_CHECK(cudaMemsetAsync(xv, 0, N * sizeof(T), c->stream));   // cg.jl:47
    if ((rc = exchange(xv, sg.nloc(), true, true))) return rc;              // halo planes of the new x
    *iters = h->iter;
    *relres = h->relres;
    *flag = h->flag;
    return SIPB_OK;
  }
  // bytes of the loop iterations that ran (launches queued behind `done` return immediately and move nothing)
  void account_cg_loops(const CgState* h) {
    sipb_ctx* c = ctx;
    const double vecN = (double)N * sizeof(T);
    const double q_rows = q_classes ? 0.0 : (double)q_offs.size();
    c->account(KC_SPMV_DOT, h->loops * (q_rows + 2) * vecN);                          // Q, p -> Ap
    c->account(KC_CG_XR, h->loops * 6 * vecN);                                        // x, r, p, Ap -> x, r
    c->account(KC_CG_P, std::max(0, h->loops - (h->flag == 0 ? 1 : 0)) * 3 * vecN);   // r, p -> p
  }
  // a deferred (graph) CG: the state arrived with the per-iteration scalars
  void finish_cg(int* iters, double* relres, int* flag) {
    sipb_ctx* c = ctx;
    const CgState* h = c->h_cg;
    account_cg_loops(h);
    // kernels the graph ran: prologue (2), three per iteration, the zero-fill check
    c->launches[KC_SPMV_DOT] += h->loops; c->launches[KC_CG_XR] += h->loops; c->launches[KC_CG_P] += h->loops;
    c->launches[KC_CG_INIT] += 1; c->launches[KC_CG_FIN] += 1;
    c->total_launches += 3 * (int64_t)h->loops + 2;
    *iters = h->iter;
    *relres = h->relres;
    *flag = h->flag;
  }

  int solve(const void* m_h, void* x_h, void* const* l_h, void* const* y_h, const sipb_options* o,
            sipb_log* log) override;
  // the two vector phases of one PARSDMM iteration (solve runs them around the CG; sipb_iter_probe runs them alone)
  int rhs_phase(int i, const std::vector<T>& rho, bool fuse_rdual);
  int yl_phase(int i, const std::vector<T>& rho, const std::vector<T>& gamma, bool do_adapt, bool fuse_stop,
               bool fuse_rdual);
};

// ---------------------------------------------------------------------------------------------
// scalar logic in TF arithmetic
// ---------------------------------------------------------------------------------------------
template <typename T>
static void adapt_scalar(const double* sm, T& rho, T& gamma, bool adjust_rho, bool adjust_gamma) {
  // adapt_rho_gamma.jl:31-126
  const T safeguard = (sizeof(T) == 8) ? (T)1e-10 : (T)1e-6f;
  const T eps_corr = (T)0.3;
  const T d_dHh_dlh = (T)sm[0];
  const T n_dH = (T)std::sqrt(sm[1]);
  const T n_dlh = (T)std::sqrt(sm[2]);
  const T n_dl = (T)std::sqrt(sm[3]);
  const T n_dG = (T)std::sqrt(sm[4]);
  const T d_dGh_dl = (T)sm[5];
  bool alpha_rel = false, beta_rel = false;
  T alpha_corr = 0, beta_corr = 0;
  if ((n_dH * n_dlh) > safeguard && (n_dH * n_dH) > safeguard && d_dHh_dlh > safeguard) {
    alpha_rel = true;
    alpha_corr = d_dHh_dlh / (n_dH * n_dlh);
  }
  if ((n_dG * n_dl) > safeguard && (n_dG * n_dG) > safeguard && d_dGh_dl > safeguard) {
    beta_rel = true;
    beta_corr = d_dGh_dl / (n_dG * n_dl);
  }
  bool alpha_comp = false, beta_comp = false;
  T alpha_hat = 0, beta_hat = 0;
  if (alpha_rel && alpha_corr > eps_corr) {
    alpha_comp = true;
    const T mg = d_dHh_dlh / (n_dH * n_dH);
    const T sd = (n_dlh * n_dlh) / d_dHh_dlh;
    alpha_hat = ((T)2.0 * mg > sd) ? mg : sd - mg / (T)2.0;
  }
  if (beta_rel && beta_corr > eps_corr) {
    beta_comp = true;
    const T mg = d_dGh_dl / (n_dG * n_dG);
    const T sd = (n_dl * n_dl) / d_dGh_dl;
    beta_hat = ((T)2.0 * mg > sd) ? mg : sd - mg / (T)2.0;
  }
  if (adjust_rho) {
    if (alpha_comp && beta_comp) rho = std::sqrt(alpha_hat * beta_hat);
    else if (alpha_comp) rho = alpha_hat;
    else if (beta_comp) rho = beta_hat;
  }
  if (adjust_gamma) {
    if (alpha_comp && beta_comp)
      gamma = (T)1.0 + (((T)2.0 * std::sqrt(alpha_hat * beta_hat)) / (alpha_hat + beta_hat));
    else if (alpha_comp) gamma = (T)1.9;
    else if (beta_comp) gamma = (T)1.1;
    else gamma = (T)1.5;
  }
}

static inline double jl_maximum(const double* a, int n, int stride = 1) {
  double m = -std::numeric_limits<double>::infinity();
  for (int i = 0; i < n; ++i) {
    const double v = a[(size_t)i * stride];
    if (v != v) return v;
    if (v > m) m = v;
  }
  return m;
}

// rhs = sum_i A_i'(rho_i y_i + l_i) of iteration i (rhs_compose.jl); fuse_rdual: from the second iteration on the
// gather also reduces the dual residual of iteration i-1 into the global slots 8.. (one per set)
template <typename T>
int Problem<T>::rhs_phase(int i, const std::vector<T>& rho, bool fuse_rdual) {
  sipb_ctx* c = ctx;
  const int p = (int)sets.size();
  {
    // sets are processed in the reference's order; runs of stencil sets go through one gather kernel each,
    // explicit sparse operators through k_sparse_adjoint in between (rhs += A_i'(rho_i y_i + l_i))
    const i64 ngrp = (N + 2 * Vec<T>::W - 1) / (2 * Vec<T>::W);
    const int g_rhs = (fuse_rdual && i >= 2) ? c->grid_fit((const void*)k_rhs<T, true>, ngrp)
                                             : c->grid_fit((const void*)k_rhs<T, false>, ngrp);
    bool first = true;
    int s0 = 0;
    while (s0 < p) {
      if (sets[s0]->is_sparse) {
        SetT<T>& S = *sets[s0];
        LAUNCH(c, KC_RHS, k_sparse_adjoint<T>, c->grid_for(N), S.sparse.ref(), rho[s0], (const T*)S.y.p, (const T*)S.l.p,
               rhs.p, first ? 0 : 1);
        first = false;
        ++s0;
        continue;
      }
      int s1 = s0;
      while (s1 < p && !sets[s1]->is_sparse) ++s1;
      RhsArgs<T> ra;
      memset(&ra, 0, sizeof(ra));
      ra.nsets = s1 - s0;
      ra.n[0] = (unsigned)n[0]; ra.n[1] = (unsigned)n[1]; ra.n[2] = (unsigned)n[2];
      ra.npts = npts; ra.ncols = N; ra.rhs = rhs.p;
      ra.accumulate = first ? 0 : 1;
      double rows = 0;
      for (int s = s0; s < s1; ++s) {
        ra.sets[s - s0].op = sets[s]->op;
        ra.sets[s - s0].y = sets[s]->y.p;
        ra.sets[s - s0].l = sets[s]->l.p;
        ra.sets[s - s0].y_old = sets[s]->y_old.p;
        ra.sets[s - s0].rho = rho[s];
        rows += (double)sets[s]->M;
      }
      c->account(KC_RHS, ((fuse_rdual && i >= 2 ? 3 : 2) * rows + (double)N) * sizeof(T));   // y, l (, y_old) -> rhs
      // from the second iteration on the gather also yields the dual residual of iteration i-1
      if (fuse_rdual && i >= 2)
        LAUNCH(c, KC_RHS, (k_rhs<T, true>), g_rhs, ra, c->rs, c->d_scal + kSlotGlobal + 8);
      else
        LAUNCH(c, KC_RHS, (k_rhs<T, false>), g_rhs, ra, c->rs, (double*)nullptr);
      first = false;
      s0 = s1;
    }
  }
  return SIPB_OK;
}

// y / l update of iteration i for every set (update_y_l.jl), fused with the rho/gamma adaptation sums and snapshots,
// the in-loop feasibility (every 10th iteration) and the stop sums; then the unfused dual residual, the slab halos of
// y and l and, when no distance term reduced them, the stop sums (k_stop).  Results land in the scalar slots.
template <typename T>
int Problem<T>::yl_phase(int i, const std::vector<T>& rho, const std::vector<T>& gamma, bool do_adapt, bool fuse_stop,
                         bool fuse_rdual) {
  sipb_ctx* c = ctx;
  const int p = (int)sets.size();
  const bool feas_it = (i % 10 == 0);
  const bool fuse_adapt = (i == 1) || do_adapt;
  YlMultiArgs<T>& ym = yl_multi;
  int n_multi = 0, g_multi = 1;
  auto flush_multi = [&]() {
    if (n_multi == 0) return;
    const dim3 grid((unsigned)g_multi, (unsigned)n_multi);
    if (fuse_adapt) LAUNCH(c, KC_YL_FUSED, (k_yl_multi<T, true>), grid, ym, c->rs_multi);
    else LAUNCH(c, KC_YL_FUSED, (k_yl_multi<T, false>), grid, ym, c->rs_multi);
    n_multi = 0;
    g_multi = 1;
  };
  for (int s = 0; s < p; ++s) {
    SetT<T>& S = *sets[s];
    const bool is_dist = S.desc.set_kind == SIPB_SET_DISTANCE;
    const bool want_feas = feas_it && !is_dist;
    // copy!(y_old, y) (update_y_l.jl:64) without moving data: the two buffers trade places and the
    // kernels read y^{k} from y_old while writing y^{k+1}
    S.y.swap(S.y_old);
    YlArgs<T> ya;
    memset(&ya, 0, sizeof(ya));
    ya.op = S.op;
    ya.P = proj_static(S, rho[s]);
    ya.x = x.p; ya.y = S.y.p; ya.l = S.l.p; ya.y_old = S.y_old.p; ya.s = S.s.p;
    if (S.is_sparse) {       // s = A x by the sparse kernel; the fused kernels then apply the identity to it
      LAUNCH(c, KC_OP_APPLY, k_sparse_forward<T>, c->grid_for(S.M), S.sparse.ref(), (const T*)x.p, S.s.p);
      ya.x = S.s.p;
    }
    ya.lhat0 = S.lhat0.p; ya.s0 = S.s0.p; ya.l0 = S.l0.p; ya.y0 = S.y0.p;
    ya.rho = rho[s]; ya.gamma = gamma[s];
    ya.do_sums = (do_adapt && i > 1) ? 1 : 0;     // i == 1: snapshot only (all deltas are zero)
    ya.do_snapshot = fuse_adapt ? 1 : 0;
    const int base = s * kSlotPerSet;
    const i64 nvecM = (S.M + Vec<T>::W - 1) / Vec<T>::W;
    const int g = proj_is_elementwise(S.desc.set_kind)
                      ? (fuse_adapt ? c->grid_fit((const void*)k_yl_multi<T, true>, nvecM)
                                    : c->grid_fit((const void*)k_yl_multi<T, false>, nvecM))
                      : c->grid_for(nvecM);
    // streams of M rows: l in, y and l out, y_old in when relaxed or adapting, 4 snapshots in / out
    const double rowsB = (double)S.M * sizeof(T), colsB = (double)N * sizeof(T);
    const bool needs_yold = fuse_adapt || !(gamma[s] == (T)1);
    const double adaptB = (fuse_adapt ? 4 : 0) * rowsB + (ya.do_sums ? 4 : 0) * rowsB;
    if (proj_is_elementwise(S.desc.set_kind)) {
      if (fuse_stop && is_dist) {       // the distance term also reduces the stop sums (x, m are in registers)
        ya.x_old = x_old.p;
        ya.stop_out = c->d_scal + kSlotGlobal;
      }
      c->account(KC_YL_FUSED, colsB + (3 + (needs_yold ? 1 : 0) + (ya.stop_out ? 1 : 0)) * rowsB + adaptB);
      // element-wise sets are gathered and updated by one launch per (up to) kYlMulti sets
      ya.want_feas = want_feas ? 1 : 0;
      ym.a[n_multi] = ya;
      ym.out[n_multi] = c->d_scal + base;
      g_multi = std::max(g_multi, g);
      if (++n_multi == kYlMulti) flush_multi();
    } else {
      ya.want_feas = 0;
      // s = A x is stored only when the in-loop feasibility check reads it afterwards (every 10th iteration) or the
      // operator is an explicit sparse matrix (its s buffer IS the input of the fused kernels)
      ya.store_s = (want_feas && !S.is_sparse) ? 1 : 0;
      // vector-mode cardinality on one GPU: the first levels of the radix select ride on pass 1 (k_yl_spec)
      const bool spec = S.desc.set_kind == SIPB_SET_CARDINALITY && !sg.on && c->sel_spec;
      // l1 ball on one GPU: pass 2 recomputes v, so pass 1 need not store it while the ball is inactive (the previous
      // iteration's sum|v| <= tau is the guess; a wrong guess costs the gated launch below, never the result)
      if (S.desc.set_kind == SIPB_SET_L1 && !sg.on && (c->l1_skipv == 2 || (c->l1_skipv == 1 && S.l1_inactive_prev)))
        ya.skip_v = 1;
      if (spec)
        LAUNCH(c, KC_YL_PASS1, (k_yl_spec<T>), c->grid_fit((const void*)k_yl_spec<T>, nvecM), ya, c->rs,
               c->d_scal + base + 10, &c->d_sel->spec_above, c->d_sel->spec, (const ProjParams<T>*)S.pp_y.p);
      else
        LAUNCH(c, KC_YL_PASS1, (k_yl<T, 1, false>), c->grid_fit((const void*)k_yl<T, 1, false>, nvecM), ya, c->rs,
               c->d_scal + base + 10);
      if (ya.skip_v) {
        // v was not stored: the threshold search reads it only when sum|v| > tau.  A second launch of pass 1, gated on the
        // device by that test (the statistics are in place), writes it then; it returns at once otherwise.
        YlArgs<T> yb = ya;
        yb.skip_v = 0;
        yb.store_s = 0;
        yb.gate = c->d_scal + base + 10;
        yb.gate_tau = (double)(T)S.desc.max;
        LAUNCH(c, KC_YL_PASS1, (k_yl<T, 1, false>), c->grid_fit((const void*)k_yl<T, 1, false>, nvecM), yb, c->rs,
               c->d_scal + base + 13);
      }
      // pass 1: x, l (, y_old) -> v (, s);   pass 2: v, x, l (, y_old) -> y, l
      // (an l1 set's pass 2 recomputes v instead of reading it; pass 1 skips the store while the ball is inactive)
      const int l1set = S.desc.set_kind == SIPB_SET_L1 ? 1 : 0;
      c->account(KC_YL_PASS1, colsB + (2 - ya.skip_v + (!(gamma[s] == (T)1) ? 1 : 0) + ya.store_s) * rowsB);
      c->account(KC_YL_PASS2, colsB + (4 - l1set + (needs_yold ? 1 : 0)) * rowsB + adaptB);
      i64 tie_chunk = 0;
      const bool defer = S.desc.set_kind == SIPB_SET_CARDINALITY && !sg.on && c->sel_spec;
      int rc = projector_params(S, S.y.p, base + 10, S.pp_y.p, S.warm.p, true, spec, defer ? &tie_chunk : nullptr);
      if (rc) return rc;
      ya.dyn = S.pp_y.p;
      if (tie_chunk > 0) { ya.P.tie_base = c->d_tie_base; ya.P.tie_chunk = tie_chunk; }
      if (fuse_adapt)
        LAUNCH(c, KC_YL_PASS2, (k_yl<T, 2, true>), c->grid_fit((const void*)k_yl<T, 2, true>, nvecM), ya, c->rs,
               c->d_scal + base);
      else
        LAUNCH(c, KC_YL_PASS2, (k_yl<T, 2, false>), c->grid_fit((const void*)k_yl<T, 2, false>, nvecM), ya, c->rs,
               c->d_scal + base);
      if (want_feas) {
        rc = feasibility_of(S, S.s.p, base + 1, true);
        if (rc) return rc;
      }
    }
  }
  flush_multi();
  if (!fuse_rdual) {
    for (int s = 0; s < p; ++s) {
      SetT<T>& S = *sets[s];
      if (S.is_sparse)
        LAUNCH(c, KC_RDUAL, k_sparse_rdual<T>, c->grid_for(N), S.sparse.ref(), (const T*)S.y.p, (const T*)S.y_old.p, c->rs,
               c->d_scal + s * kSlotPerSet + 3);
      else
        LAUNCH(c, KC_RDUAL, k_rdual<T>, c->grid_for((npts + Vec<T>::W - 1) / Vec<T>::W), S.op, (const T*)S.y.p,
               (const T*)S.y_old.p, c->rs, c->d_scal + s * kSlotPerSet + 3);
    }
  }
  { int rc = exchange_yl_halos(); if (rc) return rc; }   // slabs: halo planes for the next rhs gather
  if (!fuse_stop) {
    LAUNCH(c, KC_STOP, k_stop<T>, c->grid_for((N + Vec<T>::W - 1) / Vec<T>::W), N, npts, minkowski ? 1 : 0, (const T*)x.p,
           (const T*)x_old.p, (const T*)m.p, c->rs, c->d_scal + kSlotGlobal);
    c->account(KC_STOP, 3.0 * N * sizeof(T));                            // x, x_old, m
  }
  return SIPB_OK;
}

// =============================================================================================
// the PARSDMM loop
// =============================================================================================
template <typename T>
int Problem<T>::solve(const void* m_h, void* x_h, void* const* l_h, void* const* y_h, const sipb_options* o,
                      sipb_log* log) {
  SIPB_REQUIRE(finalized, SIPB_E_STATE, "problem not finalized");
  SIPB_REQUIRE(m_h && x_h && o && log, SIPB_E_INVALID, "null argument");
  sipb_ctx* c = ctx;
  const double t_begin = now_s();
  c->reset_accounting();
  c->profile = o->profile_kernels != 0;
  const int p = (int)sets.size();
  const int pp = feas_only ? p : p - 1;
  const int maxit = o->maxit;
  SIPB_REQUIRE(maxit >= 1, SIPB_E_INVALID, "maxit must be >= 1");
  SIPB_REQUIRE(o->n_rho_ini == 1 || o->n_rho_ini == p, SIPB_E_INVALID, "rho_ini must have 1 or p entries");
  SIPB_REQUIRE(o->rho_update_frequency >= 1, SIPB_E_INVALID, "rho_update_frequency must be >= 1");
  const bool warm_res = o->warm_resident != 0 && !o->zero_ini_guess;
  if (!o->zero_ini_guess && !warm_res) SIPB_REQUIRE(l_h && y_h, SIPB_E_INVALID, "warm start needs l and y");
  if (o->return_ly) SIPB_REQUIRE(l_h && y_h, SIPB_E_INVALID, "return_ly needs l and y");
  log->p = p; log->pp = pp; log->iters = 0; log->feas_rows = 1; log->stopped_feasible = 0;
  log->h2d_bytes = 0; log->d2h_bytes = 0;
  for (int q = 0; q < SIPB_N_PHASES; ++q) log->phase_seconds[q] = 0.0;
  // Phase times as TimerOutputs reports them (PARSDMM.jl:100,105,113,152,163,229): a CUDA event closes every phase
  // on the solver's stream; the elapsed device time between consecutive events is billed to the phase that ended
  // (host wall clock would bill the execution of asynchronously launched kernels to whichever phase synchronises).
  std::vector<std::pair<cudaEvent_t, int>>& pev = c->phase_events;
  size_t pev_used = 0;
  auto phase_mark = [&](int ph) {
    if (pev_used == pev.size()) {
      cudaEvent_t e;
      if (cudaEventCreate(&e) != cudaSuccess) return;
      pev.push_back({e, ph});
    }
    pev[pev_used].second = ph;
    cudaEventRecord(pev[pev_used].first, c->stream);
    ++pev_used;
  };
  auto phase_end = [&](int ph) { phase_mark(ph); };
  auto phase_collect = [&]() {
    for (size_t q = 1; q < pev_used; ++q) {
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, pev[q - 1].first, pev[q].first) == cudaSuccess)
        log->phase_seconds[pev[q].second] += 1e-3 * (double)ms;
    }
  };
  phase_mark(0);

  // ---------------- initialization (PARSDMM_initialize.jl) ------------------------------------
  const T feas_tol = (T)o->feas_tol, obj_tol = (T)o->obj_tol, evol_rel_tol = (T)o->evol_rel_tol;
  int rho_update_frequency = o->rho_update_frequency;
  bool adjust_rho = o->adjust_rho != 0, adjust_gamma = o->adjust_gamma != 0;
  bool adjust_feasibility_rho = o->adjust_feasibility_rho != 0;
  T gamma_ini = (T)o->gamma_ini;
  std::vector<T> rho(p), gamma(p);
  for (int i = 0; i < p; ++i) rho[i] = (T)(o->n_rho_ini == 1 ? o->rho_ini[0] : o->rho_ini[i]);

  // m (for Minkowski the feasibility check uses [m; 0], PARSDMM_initialize.jl:85-87)
  const bool resident = o->resident_io != 0;
  if (resident) {
    SIPB_REQUIRE(m_resident, SIPB_E_STATE, "resident_io needs a previous regular solve of this problem");
    SIPB_REQUIRE(o->zero_ini_guess, SIPB_E_INVALID, "resident_io requires zero_ini_guess");
  } else {
    SIPB_CUDA_CHECK(cudaMemcpyAsync(m.p, m_h, npts * sizeof(T), cudaMemcpyHostToDevice, c->stream));
    log->h2d_bytes += npts * sizeof(T);
    if (minkowski) SIPB_CUDA_CHECK(cudaMemsetAsync(m.p + npts, 0, npts * sizeof(T), c->stream));
    m_resident = true;
    { int rc = exchange(m.p, sg.nloc(), false, true); if (rc) return rc; }   // slabs: upper halo plane of m
  }
  cudaEvent_t ev0, ev1;
  SIPB_CUDA_CHECK(cudaEventCreate(&ev0));
  SIPB_CUDA_CHECK(cudaEventCreate(&ev1));
  SIPB_CUDA_CHECK(cudaEventRecord(ev0, c->stream));

  SIPB_CUDA_CHECK(cudaMemsetAsync(c->d_l1, 0, sizeof(L1State), c->stream));
  // initial feasibility  ||P(A m) - A m|| / (||A m|| + 100 eps)   (:97-99)
  const int nP = pp;   // P_sub has one entry per non-distance set
  for (int i = 0; i < nP; ++i) {
    SetT<T>& S = *sets[i];
    T* sv = S.s.p ? S.s.p : tmp.p;    // element-wise sets do not keep s: use the scratch vector
    if (S.is_sparse) LAUNCH(c, KC_OP_APPLY, k_sparse_forward<T>, c->grid_for(S.M), S.sparse.ref(), (const T*)m.p, sv);
    else LAUNCH(c, KC_OP_APPLY, k_op_forward<T>, c->grid_for(S.M), S.op, (const T*)m.p, sv);
    int rc = feasibility_of(S, sv, i * kSlotPerSet + 1);
    if (rc) return rc;
  }
  { int rc = ctx_sync_scalars(c); if (rc) return rc; }
  std::vector<double> feas0(std::max(nP, 1), 0.0);
  const T eps100 = (T)100 * (T)Eps<T>::v;
  for (int i = 0; i < nP; ++i) {
    const T num = (T)std::sqrt(c->h_scal[i * kSlotPerSet + 1]);
    const T den = (T)std::sqrt(c->h_scal[i * kSlotPerSet + 2]);
    feas0[i] = (double)(num / (den + eps100));
  }
  for (int i = 0; i < nP; ++i) log->set_feasibility[i] = feas0[i];
  bool stop = nP > 0 && (T)jl_maximum(feas0.data(), nP) < feas_tol;   // :101-104
  if (o->fixed_iterations > 0) stop = false;

  for (int i = 0; i < pp; ++i)                                     // :107-114
    if (sets[i]->desc.ncvx) { rho_update_frequency = 3; adjust_gamma = false; gamma_ini = (T)0.75; }
  for (int i = 0; i < p; ++i) gamma[i] = gamma_ini;

  if (stop) {                                                      // PARSDMM.jl:63-82
    // x = m (Minkowski: [m; 0]); device buffer m already holds exactly that.  The resident state must equal what
    // is returned — a later sipb_problem_warm_from (multilevel) reads x, l, y from these buffers: x = m, and
    // l = y = 0 for a zero start (PARSDMM_initialize.jl:304-313) or the caller's l, y otherwise.
    SIPB_CUDA_CHECK(cudaMemcpyAsync(x.p, m.p, N * sizeof(T), cudaMemcpyDeviceToDevice, c->stream));
    if (o->zero_ini_guess) {
      for (auto& S : sets) {
        SIPB_CUDA_CHECK(cudaMemsetAsync(S->y.p, 0, S->M * sizeof(T), c->stream));
        SIPB_CUDA_CHECK(cudaMemsetAsync(S->l.p, 0, S->M * sizeof(T), c->stream));
      }
    } else if (!warm_res && l_h && y_h) {
      for (int i = 0; i < p; ++i) {
        if (!l_h[i] || !y_h[i]) continue;
        SIPB_CUDA_CHECK(cudaMemcpyAsync(sets[i]->l.p, l_h[i], sets[i]->M * sizeof(T), cudaMemcpyHostToDevice, c->stream));
        SIPB_CUDA_CHECK(cudaMemcpyAsync(sets[i]->y.p, y_h[i], sets[i]->M * sizeof(T), cudaMemcpyHostToDevice, c->stream));
      }
    }
    if (!resident) {
      SIPB_CUDA_CHECK(cudaMemcpyAsync(x_h, m.p, N * sizeof(T), cudaMemcpyDeviceToHost, c->stream));
      log->d2h_bytes += N * sizeof(T);
    }
    SIPB_CUDA_CHECK(cudaStreamSynchronize(c->stream));
    cudaEventDestroy(ev0);
    cudaEventDestroy(ev1);
    log->stopped_feasible = 1;
    log->iters = 0;
    log->feas_rows = 1;
    log->total_launches = c->total_launches;
    c->collect_profile();
    for (int q = 0; q < SIPB_N_KERNEL_CLASSES; ++q) {
      log->kernel_launches[q] = c->launches[q];
      log->kernel_ms[q] = c->ms[q];
      log->kernel_bytes[q] = c->bytes[q];
    }
    phase_end(0);
    SIPB_CUDA_CHECK(cudaStreamSynchronize(c->stream));
    phase_collect();
    log->solve_seconds = now_s() - t_begin;
    log->device_seconds = 0.0;
    return SIPB_OK;
  }

  // start vectors (:304-313 zero guess, otherwise the caller's x,l,y)
  if (o->zero_ini_guess) {
    SIPB_CUDA_CHECK(cudaMemsetAsync(x.p, 0, N * sizeof(T), c->stream));
    for (auto& S : sets) {
      SIPB_CUDA_CHECK(cudaMemsetAsync(S->y.p, 0, S->M * sizeof(T), c->stream));
      SIPB_CUDA_CHECK(cudaMemsetAsync(S->l.p, 0, S->M * sizeof(T), c->stream));
    }
  } else if (!warm_res) {
    SIPB_CUDA_CHECK(cudaMemcpyAsync(x.p, x_h, N * sizeof(T), cudaMemcpyHostToDevice, c->stream));
    log->h2d_bytes += N * sizeof(T);
    for (int i = 0; i < p; ++i) {
      SetT<T>& S = *sets[i];
      SIPB_REQUIRE(l_h[i] && y_h[i], SIPB_E_INVALID, "warm start needs every l[i], y[i]");
      SIPB_CUDA_CHECK(cudaMemcpyAsync(S.l.p, l_h[i], S.M * sizeof(T), cudaMemcpyHostToDevice, c->stream));
      SIPB_CUDA_CHECK(cudaMemcpyAsync(S.y.p, y_h[i], S.M * sizeof(T), cudaMemcpyHostToDevice, c->stream));
      log->h2d_bytes += 2 * S.M * sizeof(T);
    }
  }
  for (auto& S : sets) {
    // the 16 work vectors per set of PARSDMM_initialize.jl:158-184 collapse to 7 (8 for reduction-type
    // projectors): x_hat, r_pri, l_hat, l_old, d_* are register temporaries of the fused kernel
    for (DevBuf<T>* b : {&S->y_old, &S->s, &S->s0, &S->y0, &S->l0, &S->lhat0})
      if (b->p) SIPB_CUDA_CHECK(cudaMemsetAsync(b->p, 0, S->M * sizeof(T), c->stream));
    SIPB_CUDA_CHECK(cudaMemsetAsync(S->warm.p, 0, 2 * sizeof(double), c->stream));
  }
  SIPB_CUDA_CHECK(cudaMemsetAsync(x_old.p, 0, N * sizeof(T), c->stream));
  if (sg.on) {      // halo planes of the start vectors
    int rc = exchange(x.p, sg.nloc(), true, true);
    if (rc) return rc;
    for (auto& S : sets)
      if (S->z_halo) SIPB_CUDA_CHECK(cudaMemsetAsync(S->y_old.p - sg.plane, 0, sg.plane * sizeof(T), c->stream));
    rc = exchange_yl_halos();
    if (rc) return rc;
  }

  // Q = sum rho_i AtA_i, accumulated set by set, diagonal by diagonal (:223-229)
  if (q_classes) SIPB_CUDA_CHECK(cudaMemsetAsync(Q_tab.p, 0, (size_t)kMaxClasses * q_offs.size() * sizeof(T), c->stream));
  else SIPB_CUDA_CHECK(cudaMemsetAsync(Q.p, 0, (size_t)ld * q_offs.size() * sizeof(T), c->stream));
  for (int i = 0; i < p; ++i) q_add(*sets[i], rho[i]);
  // reset tolerance memory (x_solve_tol_ref = TF(1.0), PARSDMM.jl:93)
  c->h_cg->tol_prev = 1.0;
  SIPB_CUDA_CHECK(cudaMemcpyAsync(&c->d_cg->tol_prev, &c->h_cg->tol_prev, sizeof(double), cudaMemcpyHostToDevice, c->stream));

  int ind_ref = maxit;                                             // PARSDMM_initialize.jl:30
  int counter = 2;                                                 // PARSDMM.jl:91
  const int p_log = p;
  auto LG = [&](double* arr, int it, int col, int ncol) -> double& { return arr[(size_t)it * ncol + col]; };
  phase_end(0);

  int last_cg = 1;
  int iters_done = 0;
  bool any_sparse = false;
  for (auto& S : sets) any_sparse = any_sparse || S->is_sparse;
  // obj / evol_x sums (PARSDMM.jl:140-145): reduced by the distance term's y/l update when there is one
  const bool fuse_stop = !feas_only && !minkowski && getenv("SIPB_FUSE_STOP_OFF") == nullptr;
  const bool fuse_rdual = p <= kRdualSets && !any_sparse;
  const int it_limit = o->fixed_iterations > 0 ? std::min(o->fixed_iterations, maxit) : maxit;
  for (int i = 1; i <= it_limit; ++i) {
    // ---------------- rhs (rhs_compose.jl) ---------------------------------------------------
    { int rc = rhs_phase(i, rho, fuse_rdual); if (rc) return rc; }
    phase_end(1);
    // ---------------- x-minimisation (argmin_x.jl + cg.jl) -----------------------------------
    int cg_it = 0, cg_flag = 0;
    double cg_relres = 0.0;
    bool cg_deferred = false;
    {
      // device-side loop (one graph launch, no host poll) unless the kernel table is being profiled or the slabs
      // use NCCL inside the CG
      const bool loop_on_device = c->graph_loops && !c->profile && (!sg.on || r_shared != nullptr);
      int rc = run_cg(rhs.p, x.p, x_old.p, i, 0.0, 1000, last_cg + 1, &cg_it, &cg_relres, &cg_flag,
                      loop_on_device ? &cg_deferred : nullptr);
      if (rc) return rc;
      last_cg = cg_it;
    }
    log->cg_it[i - 1] = cg_it;
    log->cg_relres[i - 1] = cg_relres;
    phase_end(2);
    // ---------------- y / l update (update_y_l.jl) --------------------------------------------
    const bool feas_it = (i % 10 == 0);
    // rho/gamma adaptation is fused into the y/l kernels: the flags are known before the update; if
    // stop_PARSDMM switches adaptation off in this very iteration the sums are simply discarded
    const bool do_adapt = (adjust_rho || adjust_gamma) && (i % rho_update_frequency == 0);
    { int rc = yl_phase(i, rho, gamma, do_adapt, fuse_stop, fuse_rdual); if (rc) return rc; }
    { int rc = ctx_sync_scalars(c, true); if (rc) return rc; }
    if (c->p2p) SIPB_REQUIRE(*c->h_p2p_err == 0, SIPB_E_NCCL, "peer-memory collective timed out (a rank stopped participating)");
    SIPB_REQUIRE(!c->h_l1->failed, SIPB_E_STATE, "l1 threshold search did not converge");
    if (cg_deferred) {
      finish_cg(&cg_it, &cg_relres, &cg_flag);
      last_cg = cg_it;
      log->cg_it[i - 1] = cg_it;
      log->cg_relres[i - 1] = cg_relres;
    }
    {
      T rp_tot = 0, rd_tot = 0;
      for (int s = 0; s < p; ++s) {
        const int base = s * kSlotPerSet;
        const T rp = (T)std::sqrt(c->h_scal[base + 0]);            // update_y_l.jl:81
        LG(log->r_pri, i - 1, s, p_log) = (double)rp;
        if (sets[s]->desc.set_kind == SIPB_SET_L1 && !sg.on)       // k_l1_begin's test on this iteration's sum|v|
          sets[s]->l1_inactive_prev = (T)c->h_scal[base + 10] <= (T)sets[s]->desc.max;
        rp_tot = rp_tot + rp;
        if (!fuse_rdual) {
          const T rd = rho[s] * (T)std::sqrt(c->h_scal[base + 3]);   // :84
          LG(log->r_dual, i - 1, s, p_log) = (double)rd;
          rd_tot = rd_tot + rd;
        }
        if (feas_it && s < pp) {                                   // :90-94
          const T num = (T)std::sqrt(c->h_scal[base + 1]);
          const T den = (T)std::sqrt(c->h_scal[base + 2]);
          LG(log->set_feasibility, counter - 1, s, pp) = (double)(num / (den + eps100));
        }
      }
      if (feas_it) counter += 1;                                   // :103-105
      if (!fuse_rdual) {
        log->r_dual_total[i - 1] = (double)rd_tot;                 // PARSDMM.jl:134
      } else if (i >= 2) {
        // r_dual of iteration i-1 arrived with this iteration's rhs kernel (it is log-only: no rule reads it)
        T tot = 0;
        for (int s = 0; s < p; ++s) {
          const T rd = (T)LG(log->rho, i - 2, s, p_log) * (T)std::sqrt(c->h_scal[kSlotGlobal + 8 + s]);
          LG(log->r_dual, i - 2, s, p_log) = (double)rd;
          tot = tot + rd;
        }
        log->r_dual_total[i - 2] = (double)tot;
      }
      log->r_pri_total[i - 1] = (double)rp_tot;                    // :138
      const double* g = c->h_scal + kSlotGlobal;
      const T nxm = (T)std::sqrt(g[0]);
      log->obj[i - 1] = (double)((T)0.5 * (nxm * nxm));            // :140/:142
      log->evol_x[i - 1] = (double)((T)std::sqrt(g[1]) / (T)std::sqrt(g[2]));   // :145
      for (int s = 0; s < p; ++s) {
        LG(log->rho, i - 1, s, p_log) = (double)rho[s];
        LG(log->gamma, i - 1, s, p_log) = (double)gamma[s];
      }
    }
    iters_done = i;
    phase_end(3);
    // ---------------- stopping rules (stop_PARSDMM.jl:23-52) ---------------------------------
    if (o->fixed_iterations <= 0) {
      bool stp = false;
      if (i > 6) {
        double relmax = -std::numeric_limits<double>::infinity();
        bool nan = false;
        for (int q = i - 6; q < i; ++q) {   // 0-based rows i-6..i-1 vs previous
          const T a = (T)log->obj[q], b = (T)log->obj[q - 1];
          const T rel = std::fabs((a - b) / b);
          if (rel != rel) nan = true;
          if ((double)rel > relmax) relmax = (double)rel;
        }
        const double fmax = pp > 0 ? jl_maximum(log->set_feasibility + (size_t)(counter - 2) * pp, pp) : 0.0;
        if (!nan && (T)fmax < feas_tol && (T)relmax < obj_tol) stp = true;
      }
      if (i > 5) {
        const double emax = jl_maximum(log->evol_x + (i - 6), 6);
        if ((T)emax < evol_rel_tol) stp = true;
      }
      {
        const int lo = std::max(i - 50, 1);
        if (i > 20 && adjust_rho &&
            log->r_pri_total[i - 1] > jl_maximum(log->r_pri_total + (lo - 1), (i - 1) - (lo - 1))) {
          adjust_rho = false; adjust_feasibility_rho = false; adjust_gamma = false;
          ind_ref = i;
        }
        const int lo2 = std::max(ind_ref, std::max(i - 50, 1));
        if (!adjust_rho && i > ind_ref + 25 &&
            log->r_pri_total[i - 1] > jl_maximum(log->r_pri_total + (lo2 - 1), (i - 1) - (lo2 - 1)))
          stp = true;
      }
      phase_end(4);
      if (stp) break;
    }
    // ---------------- rho / gamma adaptation (PARSDMM.jl:164-226) ----------------------------
    // the reductions were produced by the fused y/l kernels of this iteration (h_scal already synced)
    if ((adjust_rho || adjust_gamma) && (i % rho_update_frequency == 0)) {
      static const double zeros6[6] = {0, 0, 0, 0, 0, 0};
      for (int s = 0; s < p; ++s)
        adapt_scalar<T>(i > 1 ? c->h_scal + s * kSlotPerSet + 4 : zeros6, rho[s], gamma[s], adjust_rho, adjust_gamma);
    }
    if (adjust_feasibility_rho && i % 10 == 0 && i > 10 && pp > 0) {       // :213-223
      const double* row = log->set_feasibility + (size_t)(counter - 2) * pp;
      int idx = 0;
      bool have_nan = false;
      for (int s = 0; s < pp; ++s) {
        if (row[s] != row[s]) { if (!have_nan) { idx = s; have_nan = true; } }
        else if (!have_nan && row[s] > row[idx]) idx = s;
      }
      rho[idx] = (T)2.0 * rho[idx];
    }
    for (int s = 0; s < p; ++s) {                                           // :226
      T v = rho[s];
      v = (v != v) ? v : (v < (T)1e4 ? v : (T)1e4);
      v = (v != v) ? v : (v > (T)1e-2 ? v : (T)1e-2);
      rho[s] = v;
    }
    phase_end(5);
    // ---------------- Q update (Q_update!.jl:45-49) -------------------------------------------
    for (int s = 0; s < p; ++s) {
      const T logged = (T)LG(log->rho, i - 1, s, p_log);
      if (rho[s] != logged) q_add(*sets[s], rho[s] - logged);
    }
    phase_end(6);
  }
  if (fuse_rdual && iters_done >= 1) {
    // dual residual of the last iteration (stand-alone pass)
    for (int s = 0; s < p; ++s) {
      SetT<T>& S = *sets[s];
      LAUNCH(c, KC_RDUAL, k_rdual<T>, c->grid_for((npts + Vec<T>::W - 1) / Vec<T>::W), S.op, (const T*)S.y.p,
             (const T*)S.y_old.p, c->rs, c->d_scal + s * kSlotPerSet + 3);
    }
    int rc = ctx_sync_scalars(c);
    if (rc) return rc;
    T tot = 0;
    for (int s = 0; s < p; ++s) {
      const T rd = (T)LG(log->rho, iters_done - 1, s, p_log) * (T)std::sqrt(c->h_scal[s * kSlotPerSet + 3]);
      LG(log->r_dual, iters_done - 1, s, p_log) = (double)rd;
      tot = tot + rd;
    }
    log->r_dual_total[iters_done - 1] = (double)tot;
  }
  SIPB_CUDA_CHECK(cudaEventRecord(ev1, c->stream));

  // ---------------- results -------------------------------------------------------------------
  if (!resident) {
    SIPB_CUDA_CHECK(cudaMemcpyAsync(x_h, x.p, N * sizeof(T), cudaMemcpyDeviceToHost, c->stream));
    log->d2h_bytes += N * sizeof(T);
  }
  if (o->return_ly && !resident) {
    for (int i = 0; i < p; ++i) {
      SetT<T>& S = *sets[i];
      SIPB_CUDA_CHECK(cudaMemcpyAsync(l_h[i], S.l.p, S.M * sizeof(T), cudaMemcpyDeviceToHost, c->stream));
      SIPB_CUDA_CHECK(cudaMemcpyAsync(y_h[i], S.y.p, S.M * sizeof(T), cudaMemcpyDeviceToHost, c->stream));
      log->d2h_bytes += 2 * S.M * sizeof(T);
    }
  }
  SIPB_CUDA_CHECK(cudaStreamSynchronize(c->stream));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, ev0, ev1);
  cudaEventDestroy(ev0);
  cudaEventDestroy(ev1);
  log->device_seconds = ms * 1e-3;
  phase_collect();
  log->iters = iters_done;
  log->feas_rows = counter;       // output_check_PARSDMM keeps set_feasibility[1:counter,:]
  c->collect_profile();
  log->total_launches = c->total_launches;
  for (int q = 0; q < SIPB_N_KERNEL_CLASSES; ++q) {
      log->kernel_launches[q] = c->launches[q];
      log->kernel_ms[q] = c->ms[q];
      log->kernel_bytes[q] = c->bytes[q];
    }
  log->solve_seconds = now_s() - t_begin;
  return SIPB_OK;
}

}  // namespace sipb

// =============================================================================================
// C ABI
// =============================================================================================
extern "C" {

int sipb_abi_version(void) { return SIPB_ABI_VERSION; }
const char* sipb_last_error(void) { return g_err.c_str(); }
const char* sipb_kernel_class_name(int cls) {
  return (cls >= 0 && cls < SIPB_N_KERNEL_CLASSES) ? kClassNames[cls] : "";
}

int sipb_ctx_create(int device, sipb_ctx** out) {
  SIPB_REQUIRE(out, SIPB_E_INVALID, "null out pointer");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    set_error(std::string("no CUDA device available (") + cudaGetErrorString(e) +
              "); this library has no CPU fallback");
    return SIPB_E_CUDA;
  }
  SIPB_REQUIRE(device >= 0 && device < ndev, SIPB_E_INVALID, "device index out of range");
  SIPB_CUDA_CHECK(cudaSetDevice(device));
  auto* c = new sipb_ctx();
  c->device = device;
  c->reset_accounting();
  memset(&c->cd_off, 0, sizeof(CommDev));
  memset(&c->cd_on, 0, sizeof(CommDev));
  c->cd_off.world = 1;
  cudaDeviceProp prop;
  SIPB_CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
  c->num_sms = prop.multiProcessorCount;
  SIPB_CUDA_CHECK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  SIPB_CUDA_CHECK(cudaStreamCreateWithFlags(&c->stream_body, cudaStreamNonBlocking));
  { const char* e = getenv("SIPB_GRAPH_LOOPS"); c->graph_loops = !(e && e[0] == '0'); }
  SIPB_CUDA_CHECK(cudaMalloc(&c->rs.partials, sizeof(double) * kMaxRed * kMaxBlocks));
  SIPB_CUDA_CHECK(cudaMalloc(&c->rs.counter, sizeof(unsigned int)));
  SIPB_CUDA_CHECK(cudaMemset(c->rs.counter, 0, sizeof(unsigned int)));
  SIPB_CUDA_CHECK(cudaMalloc(&c->rs_multi.partials, sizeof(double) * kMaxRed * kMaxBlocks * kYlMulti));
  SIPB_CUDA_CHECK(cudaMalloc(&c->rs_multi.counter, sizeof(unsigned int) * kYlMulti));
  SIPB_CUDA_CHECK(cudaMemset(c->rs_multi.counter, 0, sizeof(unsigned int) * kYlMulti));
  SIPB_CUDA_CHECK(cudaMalloc(&c->d_counter2, sizeof(unsigned int)));
  SIPB_CUDA_CHECK(cudaMemset(c->d_counter2, 0, sizeof(unsigned int)));
  SIPB_CUDA_CHECK(cudaMalloc(&c->d_scal, sizeof(double) * kScalSlots));
  SIPB_CUDA_CHECK(cudaMemset(c->d_scal, 0, sizeof(double) * kScalSlots));
  SIPB_CUDA_CHECK(cudaMallocHost(&c->h_scal, sizeof(double) * kScalSlots));
  SIPB_CUDA_CHECK(cudaMalloc(&c->d_cg, sizeof(CgState)));
  SIPB_CUDA_CHECK(cudaMemset(c->d_cg, 0, sizeof(CgState)));
  SIPB_CUDA_CHECK(cudaMallocHost(&c->h_cg, sizeof(CgState)));
  memset(c->h_cg, 0, sizeof(CgState));
  SIPB_CUDA_CHECK(cudaMalloc(&c->d_l1, sizeof(L1State)));
  SIPB_CUDA_CHECK(cudaMemset(c->d_l1, 0, sizeof(L1State)));
  SIPB_CUDA_CHECK(cudaMallocHost(&c->h_l1, sizeof(L1State)));
  SIPB_CUDA_CHECK(cudaMalloc(&c->d_sel, sizeof(SelState)));
  SIPB_CUDA_CHECK(cudaMemset(c->d_sel, 0, sizeof(SelState)));
  SIPB_CUDA_CHECK(cudaMalloc(&c->d_tie_counts, sizeof(unsigned long long) * kMaxBlocks));
  SIPB_CUDA_CHECK(cudaMalloc(&c->d_tie_base, sizeof(unsigned long long) * kMaxBlocks));
  SIPB_CUDA_CHECK(cudaMalloc(&c->d_sel_table, sizeof(unsigned int) * (size_t)kMaxBlocks * kSelBins));
  if (const char* e = getenv("SIPB_SEL_SPEC")) c->sel_spec = atoi(e) != 0;
  if (const char* e = getenv("SIPB_L1_SKIPV")) c->l1_skipv = atoi(e);
  *out = c;
  return SIPB_OK;
}

int sipb_ctx_destroy(sipb_ctx* c) {
  if (!c) return SIPB_OK;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  for (auto& e : c->ev_pool) { cudaEventDestroy(e.first); cudaEventDestroy(e.second); }
  for (auto& e : c->phase_events) cudaEventDestroy(e.first);
  cudaFree(c->rs.partials); cudaFree(c->rs.counter); cudaFree(c->rs_multi.partials); cudaFree(c->rs_multi.counter); cudaFree(c->d_counter2); cudaFree(c->d_scal);
  cudaFreeHost(c->h_scal); cudaFree(c->d_cg); cudaFreeHost(c->h_cg); cudaFree(c->d_l1); cudaFreeHost(c->h_l1);
  cudaFree(c->d_sel); cudaFree(c->d_tie_counts); cudaFree(c->d_sel_table); cudaFree(c->d_tie_base);
  for (int q = 0; q < kMaxRanks; ++q)
    if (c->peer_mail_base[q]) cudaIpcCloseMemHandle(c->peer_mail_base[q]);
  for (void* b : c->shared_bufs) cudaFree(b);
  for (int q = 0; q < kMaxRanks; ++q)
    if (c->peer_big_base[q]) cudaIpcCloseMemHandle(c->peer_big_base[q]);
  if (c->d_big) { cudaFree(c->d_big); cudaFree(c->bd.seq); }
  if (c->d_mail) cudaFree(c->d_mail);
  if (c->d_seq_pv) cudaFree(c->d_seq_pv);
  if (c->d_p2p_err) cudaFree(c->d_p2p_err);
  if (c->h_p2p_err) cudaFreeHost(c->h_p2p_err);
  if (c->d_gather) cudaFree(c->d_gather);
  if (c->d_gather_local) cudaFree(c->d_gather_local);
  if (c->comm) NCCL(CommDestroy)(c->comm);
  cudaStreamDestroy(c->stream);
  if (c->stream_body) cudaStreamDestroy(c->stream_body);
  delete c;
  return SIPB_OK;
}

int sipb_ctx_num_sms(sipb_ctx* c, int* out) {
  SIPB_REQUIRE(c && out, SIPB_E_INVALID, "null argument");
  *out = c->num_sms;
  return SIPB_OK;
}

// Peer-memory set-up: export this rank's mailbox with CUDA IPC, import everybody else's.  Any failure (no P2P
// between the devices, IPC unavailable, SIPB_P2P=0) turns the peer path off on ALL ranks (min-reduction of
// the success flag) and the NCCL path is used instead.
static int comm_setup_p2p(sipb_ctx* c) {
  memset(&c->cd_off, 0, sizeof(CommDev));
  memset(&c->cd_on, 0, sizeof(CommDev));
  c->cd_off.rank = c->rank;
  c->cd_off.world = c->world;
  const char* env = getenv("SIPB_P2P");
  int ok = (env && env[0] == '0') ? 0 : 1;
  if (c->world > kMaxRanks) ok = 0;
  cudaIpcMemHandle_t mine;
  memset(&mine, 0, sizeof(mine));
  if (ok) {
    ok = cudaMalloc(&c->d_mail, sizeof(PeerMail)) == cudaSuccess && cudaMemset(c->d_mail, 0, sizeof(PeerMail)) == cudaSuccess &&
         cudaMalloc(&c->d_seq_pv, 3 * sizeof(unsigned long long)) == cudaSuccess &&
         cudaMemset(c->d_seq_pv, 0, 3 * sizeof(unsigned long long)) == cudaSuccess &&
         cudaMalloc(&c->d_p2p_err, sizeof(int)) == cudaSuccess && cudaMemset(c->d_p2p_err, 0, sizeof(int)) == cudaSuccess &&
         cudaMallocHost(&c->h_p2p_err, sizeof(int)) == cudaSuccess &&
         cudaIpcGetMemHandle(&mine, c->d_mail) == cudaSuccess;
    cudaGetLastError();
  }
  std::vector<cudaIpcMemHandle_t> all(c->world);
  int rc = c->allgather_bytes(&mine, all.data(), sizeof(mine));
  if (rc) return rc;
  c->cd_on = c->cd_off;
  if (ok) {
    for (int q = 0; q < c->world && ok; ++q) {
      if (q == c->rank) { c->cd_on.mail[q] = c->d_mail; continue; }
      void* ptr = nullptr;
      if (cudaIpcOpenMemHandle(&ptr, all[q], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { ok = 0; cudaGetLastError(); break; }
      c->peer_mail_base[q] = ptr;
      c->cd_on.mail[q] = reinterpret_cast<PeerMail*>(ptr);
    }
  }
  // agree on the outcome
  double flag = ok ? 0.0 : 1.0;
  SIPB_CUDA_CHECK(cudaMemcpyAsync(c->d_scal, &flag, sizeof(double), cudaMemcpyHostToDevice, c->stream));
  rc = c->allreduce(c->d_scal, 1);
  if (rc) return rc;
  SIPB_CUDA_CHECK(cudaMemcpyAsync(&flag, c->d_scal, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  SIPB_CUDA_CHECK(cudaMemsetAsync(c->d_scal, 0, sizeof(double), c->stream));
  SIPB_CUDA_CHECK(cudaStreamSynchronize(c->stream));
  c->p2p = (flag == 0.0);
  if (c->p2p) {
    // second exported buffer: the small all-reduces of the y/l phase (failure here only keeps those on NCCL)
    cudaIpcMemHandle_t hb;
    memset(&hb, 0, sizeof(hb));
    int okb = cudaMalloc(&c->d_big, sizeof(PeerBig)) == cudaSuccess && cudaMemset(c->d_big, 0, sizeof(PeerBig)) == cudaSuccess &&
              cudaIpcGetMemHandle(&hb, c->d_big) == cudaSuccess;
    cudaGetLastError();
    std::vector<cudaIpcMemHandle_t> allb(c->world);
    rc = c->allgather_bytes(&hb, allb.data(), sizeof(hb));
    if (rc) return rc;
    memset(&c->bd, 0, sizeof(c->bd));
    c->bd.rank = c->rank;
    c->bd.world = c->world;
    c->bd.err = c->d_p2p_err;
    for (int q = 0; q < c->world && okb; ++q) {
      if (q == c->rank) { c->bd.box[q] = c->d_big; continue; }
      void* ptr = nullptr;
      if (cudaIpcOpenMemHandle(&ptr, allb[q], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { okb = 0; cudaGetLastError(); break; }
      c->peer_big_base[q] = ptr;
      c->bd.box[q] = reinterpret_cast<PeerBig*>(ptr);
    }
    double fb = okb ? 0.0 : 1.0;       // all ranks or none (plain NCCL: d_big is not in use yet)
    SIPB_CUDA_CHECK(cudaMemcpyAsync(c->d_scal, &fb, sizeof(double), cudaMemcpyHostToDevice, c->stream));
    c->nccl_calls++;
    SIPB_NCCL_CHECK(NCCL(AllReduce)(c->d_scal, c->d_scal, 1, ncclDouble, ncclSum, c->comm, c->stream));
    SIPB_CUDA_CHECK(cudaMemcpyAsync(&fb, c->d_scal, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    SIPB_CUDA_CHECK(cudaMemsetAsync(c->d_scal, 0, sizeof(double), c->stream));
    SIPB_CUDA_CHECK(cudaStreamSynchronize(c->stream));
    const char* envb = getenv("SIPB_PEER_ALLREDUCE");
    if (fb != 0.0 || (envb && envb[0] == '0')) {
      if (c->d_big) cudaFree(c->d_big);
      c->d_big = nullptr;           // peer_big_base mappings are closed at teardown
    } else {
      SIPB_CUDA_CHECK(cudaMalloc(&c->bd.seq, sizeof(unsigned long long)));
      SIPB_CUDA_CHECK(cudaMemset(c->bd.seq, 0, sizeof(unsigned long long)));
    }
    c->cd_on.on = 1;
    c->cd_on.has_lo = c->rank > 0;
    c->cd_on.has_hi = c->rank < c->world - 1;
    c->cd_on.err = c->d_p2p_err;
    c->cd_on.seq = c->d_seq_pv;
    c->cd_on.pv = c->d_seq_pv + 1;
    c->cd_on.bseq = c->d_seq_pv + 2;
  }
  return SIPB_OK;
}

int sipb_comm_unique_id(void* out128) {
  SIPB_REQUIRE(out128, SIPB_E_INVALID, "null argument");
  static_assert(NCCL_UNIQUE_ID_BYTES == 128, "unique id size");
  SIPB_REQUIRE(nccl_api()->ok, SIPB_E_NCCL, "libnccl.so.2 could not be loaded");
  ncclUniqueId id;
  SIPB_NCCL_CHECK(NCCL(GetUniqueId)(&id));
  memcpy(out128, &id, sizeof(id));
  return SIPB_OK;
}
int sipb_comm_init(sipb_ctx* ctx, int rank, int world, const void* uid128) {
  SIPB_REQUIRE(ctx, SIPB_E_INVALID, "null ctx");
  SIPB_REQUIRE(world >= 1 && rank >= 0 && rank < world, SIPB_E_INVALID, "bad rank / world");
  SIPB_REQUIRE(ctx->comm == nullptr, SIPB_E_STATE, "communicator already initialised");
  if (world == 1) { ctx->rank = 0; ctx->world = 1; return SIPB_OK; }
  SIPB_REQUIRE(uid128, SIPB_E_INVALID, "null unique id");
  SIPB_REQUIRE(nccl_api()->ok, SIPB_E_NCCL, "libnccl.so.2 could not be loaded");
  SIPB_CUDA_CHECK(cudaSetDevice(ctx->device));
  ncclUniqueId id;
  memcpy(&id, uid128, sizeof(id));
  SIPB_NCCL_CHECK(NCCL(CommInitRank)(&ctx->comm, world, id, rank));
  ctx->rank = rank;
  ctx->world = world;
  SIPB_CUDA_CHECK(cudaMalloc(&ctx->d_gather, sizeof(unsigned long long) * 4 * world));
  SIPB_CUDA_CHECK(cudaMalloc(&ctx->d_gather_local, sizeof(unsigned long long) * 4));
  // warm the communicator up (first collective builds the channels)
  int rc = ctx->allreduce(ctx->d_scal, kScalSlots);
  if (rc) return rc;
  SIPB_CUDA_CHECK(cudaMemsetAsync(ctx->d_scal, 0, kScalSlots * sizeof(double), ctx->stream));
  SIPB_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  return comm_setup_p2p(ctx);
}
int sipb_comm_info(sipb_ctx* ctx, int* rank, int* world) {
  SIPB_REQUIRE(ctx && rank && world, SIPB_E_INVALID, "null argument");
  *rank = ctx->rank;
  *world = ctx->world;
  return SIPB_OK;
}
int sipb_comm_peer_path(sipb_ctx* ctx, int* active) {
  SIPB_REQUIRE(ctx && active, SIPB_E_INVALID, "null argument");
  *active = ctx->p2p ? 1 : 0;
  return SIPB_OK;
}
/* plane range [k0,k1) of the slowest axis owned by `rank` (contiguous, sizes differ by at most one) */
int sipb_slab_range(int64_t n_last, int rank, int world, int64_t* k0, int64_t* k1) {
  SIPB_REQUIRE(k0 && k1 && world >= 1 && rank >= 0 && rank < world, SIPB_E_INVALID, "bad argument");
  *k0 = n_last * rank / world;
  *k1 = n_last * (rank + 1) / world;
  return SIPB_OK;
}

int sipb_problem_create(sipb_ctx* ctx, int dtype, int ndim, const int64_t* n, const double* h, int minkowski,
                        int feasibility_only, sipb_problem** out) {
  SIPB_REQUIRE(ctx && n && h && out, SIPB_E_INVALID, "null argument");
  SIPB_REQUIRE(dtype == SIPB_F32 || dtype == SIPB_F64, SIPB_E_INVALID, "dtype must be SIPB_F32 or SIPB_F64");
  SIPB_REQUIRE(ndim == 2 || ndim == 3, SIPB_E_INVALID, "ndim must be 2 or 3");
  for (int a = 0; a < ndim; ++a) SIPB_REQUIRE(n[a] >= 2, SIPB_E_INVALID, "grid dimensions must be >= 2");
  SIPB_CUDA_CHECK(cudaSetDevice(ctx->device));
  sipb_problem* pb = nullptr;
  int err = SIPB_OK;
  if (dtype == SIPB_F32) {
    auto* q = new Problem<float>(ctx, dtype, ndim, n, h, minkowski != 0, feasibility_only != 0);
    err = q->create_error;
    pb = q;
  } else {
    auto* q = new Problem<double>(ctx, dtype, ndim, n, h, minkowski != 0, feasibility_only != 0);
    err = q->create_error;
    pb = q;
  }
  if (err) {
    delete pb;
    set_error(err == SIPB_E_UNSUPPORTED
                  ? "multi-GPU slabs need a 3-D, non-Minkowski problem (2-D and Minkowski problems stay on one GPU)"
                  : "the slowest grid axis has fewer planes than there are ranks");
    return err;
  }
  *out = pb;
  return SIPB_OK;
}
int sipb_problem_add_set(sipb_problem* pb, const sipb_set_desc* d) {
  SIPB_REQUIRE(pb && d, SIPB_E_INVALID, "null argument");
  return pb->add_set(d);
}
int sipb_problem_set_ata(sipb_problem* pb, int idx, const void* R, int64_t rows, const int64_t* offs, int nd) {
  SIPB_REQUIRE(pb && R && offs, SIPB_E_INVALID, "null argument");
  return pb->set_ata(idx, R, rows, offs, nd);
}
int sipb_problem_set_ata_classes(sipb_problem* pb, int idx, const void* tab, const int64_t* offs, int nd) {
  SIPB_REQUIRE(pb && tab && offs, SIPB_E_INVALID, "null argument");
  SIPB_CUDA_CHECK(cudaSetDevice(pb->ctx->device));
  return pb->set_ata_classes(idx, tab, offs, nd);
}
int sipb_problem_finalize(sipb_problem* pb) {
  SIPB_REQUIRE(pb, SIPB_E_INVALID, "null argument");
  return pb->finalize();
}
int sipb_problem_num_q_offsets(sipb_problem* pb, int* nd) {
  SIPB_REQUIRE(pb && nd, SIPB_E_INVALID, "null argument");
  std::vector<int64_t> v;
  int rc = pb->q_offsets(v);
  if (rc) return rc;
  *nd = (int)v.size();
  return SIPB_OK;
}
int sipb_problem_q_offsets(sipb_problem* pb, int64_t* out) {
  SIPB_REQUIRE(pb && out, SIPB_E_INVALID, "null argument");
  std::vector<int64_t> v;
  int rc = pb->q_offsets(v);
  if (rc) return rc;
  for (size_t i = 0; i < v.size(); ++i) out[i] = v[i];
  return SIPB_OK;
}
int sipb_problem_q_form(sipb_problem* pb, int* form) {
  SIPB_REQUIRE(pb && form, SIPB_E_INVALID, "null argument");
  std::vector<int64_t> v;
  int rc = pb->q_offsets(v);      // fails before finalize
  if (rc) return rc;
  *form = pb->q_form();
  return SIPB_OK;
}
int sipb_problem_warm_from(sipb_problem* fine, sipb_problem* coarse, const sipb_resample_seg* segs, int nseg) {
  SIPB_REQUIRE(fine && coarse && segs && nseg >= 0, SIPB_E_INVALID, "null argument");
  SIPB_CUDA_CHECK(cudaSetDevice(fine->ctx->device));
  return fine->warm_from(coarse, segs, nseg);
}
int sipb_problem_destroy(sipb_problem* pb) {
  if (pb) {
    cudaSetDevice(pb->ctx->device);
    cudaStreamSynchronize(pb->ctx->stream);
    delete pb;
  }
  return SIPB_OK;
}
int sipb_solve(sipb_problem* pb, const void* m, void* x, void* const* l, void* const* y, const sipb_options* opt,
               sipb_log* log) {
  SIPB_REQUIRE(pb, SIPB_E_INVALID, "null problem");
  SIPB_CUDA_CHECK(cudaSetDevice(pb->ctx->device));
  return pb->solve(m, x, l, y, opt, log);
}

// B independent projections side by side (RGB channels of examples/Constraint_examples_2D.jl:221-226, PARSDMM as the
// inner projector of an outer loop, examples/Dykstra_parallel_vs_PARSDMM.jl:134,149): every problem lives in its own
// context (own stream, scratch and scalar mirrors), one host thread per problem drives it, and the GPU overlaps the
// small kernels of the different streams — a single small projection is latency bound and leaves most SMs idle.
int sipb_solve_batch(sipb_problem* const* pbs, int B, const void* const* m, void* const* x, void* const* const* l,
                     void* const* const* y, const sipb_options* opt, sipb_log* const* logs, int* rcs) {
  SIPB_REQUIRE(pbs && m && x && opt && logs && B >= 1, SIPB_E_INVALID, "null argument");
  for (int b = 0; b < B; ++b) {
    SIPB_REQUIRE(pbs[b] && m[b] && x[b] && logs[b], SIPB_E_INVALID, "null entry in the batch");
    SIPB_REQUIRE(pbs[b]->ctx->world == 1, SIPB_E_UNSUPPORTED, "batched projections run as replicas: one GPU per process");
    for (int q = 0; q < b; ++q)
      SIPB_REQUIRE(pbs[q]->ctx != pbs[b]->ctx, SIPB_E_INVALID,
                   "every problem of a batch needs its own context (sipb_ctx_create): a context owns one stream");
  }
  std::vector<int> rc(B, SIPB_OK);
  std::vector<std::string> errs(B);
  std::vector<std::thread> th;
  th.reserve(B);
  for (int b = 0; b < B; ++b) {
    th.emplace_back([&, b]() {
      if (cudaSetDevice(pbs[b]->ctx->device) != cudaSuccess) {
        rc[b] = SIPB_E_CUDA;
        errs[b] = "cudaSetDevice failed";
        return;
      }
      rc[b] = pbs[b]->solve(m[b], x[b], l ? l[b] : nullptr, y ? y[b] : nullptr, opt, logs[b]);
      if (rc[b]) errs[b] = g_err;          // thread-local message of this worker
    });
  }
  for (auto& t : th) t.join();
  int first = SIPB_OK;
  for (int b = 0; b < B; ++b) {
    if (rcs) rcs[b] = rc[b];
    if (rc[b] && !first) {
      first = rc[b];
      set_error("problem " + std::to_string(b) + " of the batch: " + errs[b]);
    }
  }
  return first;
}

int sipb_op_rows(int ndim, const int64_t* n, int op_kind, int64_t* rows) {
  SIPB_REQUIRE(n && rows, SIPB_E_INVALID, "null argument");
  const int64_t r = op_rows_host(ndim, n, op_kind);
  SIPB_REQUIRE(r >= 0, SIPB_E_UNSUPPORTED, "operator kind not available for this grid dimensionality");
  *rows = r;
  return SIPB_OK;
}

}  // extern "C"

// ---- unit entry points (templated bodies) ------------------------------------------------------
namespace sipb {

template <typename T>
static int upload_cds(sipb_ctx* c, int64_t N, int nd, const void* R, i64 ld, DevBuf<T>& d) {
  SIPB_CUDA_CHECK(d.alloc((size_t)ld * nd));
  SIPB_CUDA_CHECK(cudaMemsetAsync(d.p, 0, (size_t)ld * nd * sizeof(T), c->stream));
  SIPB_CUDA_CHECK(cudaMemcpy2DAsync(d.p, ld * sizeof(T), R, N * sizeof(T), N * sizeof(T), nd, cudaMemcpyHostToDevice,
                                    c->stream));
  return SIPB_OK;
}

template <typename T>
static int cds_spmv_impl(sipb_ctx* c, int64_t N, int nd, const void* R, const int64_t* offs, const void* x, void* y) {
  const i64 ld = (N + 63) / 64 * 64;
  DevBuf<T> dR, dx, dy;
  int rc = upload_cds<T>(c, N, nd, R, ld, dR);
  if (rc) return rc;
  SIPB_CUDA_CHECK(dx.alloc((size_t)N));
  SIPB_CUDA_CHECK(dy.alloc((size_t)N));
  SIPB_CUDA_CHECK(cudaMemcpyAsync(dx.p, x, N * sizeof(T), cudaMemcpyHostToDevice, c->stream));
  SpmvArgs<T> a;
  a.R = dR.p; a.ld = ld; a.nd = nd;
  for (int j = 0; j < nd; ++j) a.off[j] = offs[j];
  a.N = N; a.row0 = 0; a.Nglob = N; a.x = dx.p; a.y = dy.p;
  a.x_lo = nullptr; a.x_hi = nullptr; a.n_lo = 0; a.tab = nullptr; a.fast = 0;
  LAUNCH(c, KC_SPMV, (k_spmv<T, false>), c->grid_for((N + Vec<T>::W - 1) / Vec<T>::W), a, c->rs, (double*)nullptr,
         (const int*)nullptr, c->cd_off);
  SIPB_CUDA_CHECK(cudaGetLastError());
  SIPB_CUDA_CHECK(cudaMemcpyAsync(y, dy.p, N * sizeof(T), cudaMemcpyDeviceToHost, c->stream));
  SIPB_CUDA_CHECK(cudaStreamSynchronize(c->stream));
  return SIPB_OK;
}

// minimal stand-alone problem wrapper so that sipb_cds_cg can reuse Problem<T>::run_cg
template <typename T>
static int cds_cg_impl(sipb_ctx* c, int64_t N, int nd, const void* R, const int64_t* offs, const void* b, void* x,
                       double tol, int max_iter, int* flag, double* relres, int* iters) {
  int64_t nn[3] = {N, 1, 1};
  double hh[3] = {1, 1, 1};
  Problem<T> P(c, sizeof(T) == 4 ? SIPB_F32 : SIPB_F64, 2, nn, hh, false, true);
  P.npts = N; P.N = N; P.ld = (N + 63) / 64 * 64;
  int rc = upload_cds<T>(c, N, nd, R, P.ld, P.Q);
  if (rc) return rc;
  P.q_offs.assign(offs, offs + nd);
  DevBuf<T> db;
  SIPB_CUDA_CHECK(db.alloc((size_t)N));
  SIPB_CUDA_CHECK(P.x.alloc((size_t)N));
  SIPB_CUDA_CHECK(P.r.alloc((size_t)N));
  SIPB_CUDA_CHECK(P.pvec.alloc((size_t)N));
  SIPB_CUDA_CHECK(P.Ap.alloc((size_t)N));
  SIPB_CUDA_CHECK(cudaMemcpyAsync(db.p, b, N * sizeof(T), cudaMemcpyHostToDevice, c->stream));
  SIPB_CUDA_CHECK(cudaMemcpyAsync(P.x.p, x, N * sizeof(T), cudaMemcpyHostToDevice, c->stream));
  rc = P.run_cg(db.p, P.x.p, nullptr, 0, (double)(T)tol, max_iter, 4, iters, relres, flag);
  if (rc) return rc;
  SIPB_CUDA_CHECK(cudaGetLastError());
  SIPB_CUDA_CHECK(cudaMemcpyAsync(x, P.x.p, N * sizeof(T), cudaMemcpyDeviceToHost, c->stream));
  SIPB_CUDA_CHECK(cudaStreamSynchronize(c->stream));
  return SIPB_OK;
}

template <typename T>
static int project_impl(sipb_ctx* c, const sipb_set_desc* d, int64_t M, void* v, const void* m_vec) {
  int64_t nn[3] = {M, 2, 1};
  double hh[3] = {1, 1, 1};
  Problem<T> P(c, sizeof(T) == 4 ? SIPB_F32 : SIPB_F64, 2, nn, hh, false, true);
  SetT<T> S;
  S.desc = *d;
  S.M = M;
  S.Mglob = M;
  SIPB_CUDA_CHECK(S.s.alloc((size_t)M));
  SIPB_CUDA_CHECK(S.pp_f.alloc(1));
  SIPB_CUDA_CHECK(S.warm.alloc(2));
  SIPB_CUDA_CHECK(P.tmp.alloc((size_t)M));
  if (d->set_kind == SIPB_SET_CARD_SLICE && d->fiber_axis != 2) SIPB_CUDA_CHECK(S.perm.alloc((size_t)M));
  SIPB_CUDA_CHECK(cudaMemsetAsync(S.warm.p, 0, 2 * sizeof(double), c->stream));
  SIPB_CUDA_CHECK(cudaMemsetAsync(S.pp_f.p, 0, sizeof(ProjParams<T>), c->stream));
  SIPB_CUDA_CHECK(cudaMemcpyAsync(S.s.p, v, M * sizeof(T), cudaMemcpyHostToDevice, c->stream));
  if (d->set_kind == SIPB_SET_HISTOGRAM) { int rc = S.alloc_hist(M); if (rc) return rc; }
  if (d->set_kind == SIPB_SET_BOUNDS_VECTOR || d->set_kind == SIPB_SET_BOUNDS_FIBER || d->set_kind == SIPB_SET_HISTOGRAM) {
    SIPB_REQUIRE(d->min_vec && d->max_vec, SIPB_E_INVALID, "vector bounds need min_vec and max_vec");
    const size_t nb = d->set_kind == SIPB_SET_BOUNDS_FIBER ? (size_t)d->td_n[d->fiber_axis] : (size_t)M;
    SIPB_CUDA_CHECK(S.lo_vec.alloc(nb));
    SIPB_CUDA_CHECK(S.hi_vec.alloc(nb));
    SIPB_CUDA_CHECK(cudaMemcpyAsync(S.lo_vec.p, d->min_vec, nb * sizeof(T), cudaMemcpyHostToDevice, c->stream));
    SIPB_CUDA_CHECK(cudaMemcpyAsync(S.hi_vec.p, d->max_vec, nb * sizeof(T), cudaMemcpyHostToDevice, c->stream));
  }
  if (d->set_kind == SIPB_SET_DISTANCE) {
    SIPB_REQUIRE(m_vec, SIPB_E_INVALID, "distance prox needs m");
    SIPB_CUDA_CHECK(P.m.alloc((size_t)M));
    SIPB_CUDA_CHECK(cudaMemcpyAsync(P.m.p, m_vec, M * sizeof(T), cudaMemcpyHostToDevice, c->stream));
  }
  if (d->set_kind == SIPB_SET_L1) SIPB_REQUIRE(d->max > 0.0, SIPB_E_INVALID, "Radius of L1 ball is negative");
  ProjDev<T> PD = P.proj_static(S, (T)d->max);
  const ProjParams<T>* dyn = nullptr;
  if (!proj_is_elementwise(d->set_kind)) {
    LAUNCH(c, KC_VEC_STATS, k_vec_stats<T>, c->grid_for(M), M, S.s.p, c->rs, c->d_scal + 10);
    int rc = P.projector_params(S, S.s.p, 10, S.pp_f.p, S.warm.p, true);
    if (rc) return rc;
    dyn = S.pp_f.p;
  }
  LAUNCH(c, KC_FEAS, k_feas_dyn<T>, c->grid_for(M), M, S.s.p, (const T*)nullptr, PD, dyn, 1, c->rs, c->d_scal);
  SIPB_CUDA_CHECK(cudaGetLastError());
  SIPB_CUDA_CHECK(cudaMemcpyAsync(v, S.s.p, M * sizeof(T), cudaMemcpyDeviceToHost, c->stream));
  SIPB_CUDA_CHECK(cudaStreamSynchronize(c->stream));
  return SIPB_OK;
}

template <typename T>
static int op_apply_impl(sipb_ctx* c, int ndim, const int64_t* n, const double* h, int op_kind, int block_mode,
                         int adjoint, const void* in, void* out) {
  OpDev op;
  int rc = make_op<T>(ndim, n, h, op_kind, block_mode, &op);
  if (rc) return rc;
  const i64 nin = adjoint ? op.rows : op.cols, nout = adjoint ? op.cols : op.rows;
  DevBuf<T> di, dout;
  SIPB_CUDA_CHECK(di.alloc((size_t)nin));
  SIPB_CUDA_CHECK(dout.alloc((size_t)nout));
  SIPB_CUDA_CHECK(cudaMemcpyAsync(di.p, in, nin * sizeof(T), cudaMemcpyHostToDevice, c->stream));
  if (adjoint) LAUNCH(c, KC_OP_APPLY, k_op_adjoint<T>, c->grid_for(nout), op, (const T*)di.p, dout.p);
  else LAUNCH(c, KC_OP_APPLY, k_op_forward<T>, c->grid_for(nout), op, (const T*)di.p, dout.p);
  SIPB_CUDA_CHECK(cudaGetLastError());
  SIPB_CUDA_CHECK(cudaMemcpyAsync(out, dout.p, nout * sizeof(T), cudaMemcpyDeviceToHost, c->stream));
  SIPB_CUDA_CHECK(cudaStreamSynchronize(c->stream));
  return SIPB_OK;
}

template <typename T>
static int sparse_apply_impl(sipb_ctx* c, const sipb_sparse* A, int adjoint, const void* in, void* out) {
  SparseDev<T> sd;
  int rc = sd.upload(A, c->stream);
  if (rc) return rc;
  const i64 nin = adjoint ? A->rows : A->cols, nout = adjoint ? A->cols : A->rows;
  DevBuf<T> di, dout;
  SIPB_CUDA_CHECK(di.alloc((size_t)nin));
  SIPB_CUDA_CHECK(dout.alloc((size_t)nout));
  SIPB_CUDA_CHECK(cudaMemcpyAsync(di.p, in, nin * sizeof(T), cudaMemcpyHostToDevice, c->stream));
  if (adjoint)
    LAUNCH(c, KC_OP_APPLY, k_sparse_adjoint<T>, c->grid_for(nout), sd.ref(), (T)1, (const T*)di.p, (const T*)nullptr, dout.p, 0);
  else
    LAUNCH(c, KC_OP_APPLY, k_sparse_forward<T>, c->grid_for(nout), sd.ref(), (const T*)di.p, dout.p);
  SIPB_CUDA_CHECK(cudaGetLastError());
  SIPB_CUDA_CHECK(cudaMemcpyAsync(out, dout.p, nout * sizeof(T), cudaMemcpyDeviceToHost, c->stream));
  SIPB_CUDA_CHECK(cudaStreamSynchronize(c->stream));
  return SIPB_OK;
}

template <typename T>
static int cds_scaled_add_impl(sipb_ctx* c, int64_t N, int nd_a, void* A, const int64_t* a_off, int nd_b, const void* B,
                               const int64_t* b_off, double alpha) {
  const i64 ld = (N + 63) / 64 * 64;
  DevBuf<T> dA, dB;
  int rc = upload_cds<T>(c, N, nd_a, A, ld, dA);
  if (rc) return rc;
  rc = upload_cds<T>(c, N, nd_b, B, ld, dB);
  if (rc) return rc;
  for (int k = 0; k < nd_b; ++k) {
    int col = -1;
    for (int j = 0; j < nd_a; ++j) if (a_off[j] == b_off[k]) { col = j; break; }
    SIPB_REQUIRE(col >= 0, SIPB_E_MISSING_DIAG,
                 "attempted to update a diagonal in A in CDS storage that does not exist. A and B need to have the "
                 "same nonzero diagonals");
    LAUNCH(c, KC_Q_UPDATE, k_cds_axpy<T>, c->grid_for((N + Vec<T>::W - 1) / Vec<T>::W), N, dA.p + (size_t)col * ld,
           (const T*)(dB.p + (size_t)k * ld), (T)alpha);
  }
  SIPB_CUDA_CHECK(cudaGetLastError());
  SIPB_CUDA_CHECK(cudaMemcpy2DAsync(A, N * sizeof(T), dA.p, ld * sizeof(T), N * sizeof(T), nd_a, cudaMemcpyDeviceToHost,
                                    c->stream));
  SIPB_CUDA_CHECK(cudaStreamSynchronize(c->stream));
  return SIPB_OK;
}

// y = A x for a CDS matrix on a 3-D grid through the tiled kernel when the geometry allows (unit tests of
// spmv_tile.cuh: arbitrary values on the 7 stencil diagonals, including the entries that wrap around line / plane ends)
template <typename T>
static int cds_spmv_grid_impl(sipb_ctx* c, const int64_t* n, int nd, const void* R, const int64_t* offs, const void* x,
                              void* y, int* used_tiled) {
  const i64 N = n[0] * n[1] * n[2];
  const i64 ld = (N + 63) / 64 * 64;
  DevBuf<T> dR, dx, dy;
  int rc = upload_cds<T>(c, N, nd, R, ld, dR);
  if (rc) return rc;
  SIPB_CUDA_CHECK(dx.alloc((size_t)N));
  SIPB_CUDA_CHECK(dy.alloc((size_t)N));
  SIPB_CUDA_CHECK(cudaMemcpyAsync(dx.p, x, N * sizeof(T), cudaMemcpyHostToDevice, c->stream));
  SpmvArgs<T> a;
  memset(&a, 0, sizeof(a));
  a.R = dR.p; a.ld = ld; a.nd = nd;
  for (int j = 0; j < nd; ++j) a.off[j] = offs[j];
  a.N = N; a.row0 = 0; a.Nglob = N; a.x = dx.p; a.y = dy.p;
  a.gn[0] = (unsigned)n[0]; a.gn[1] = (unsigned)n[1]; a.gn[2] = (unsigned)n[2]; a.npts = (unsigned)N;
  const TileGeom tg = plan_tile<T>(3, n, false, std::vector<int64_t>(offs, offs + nd), n[2], 0, false, false, c->num_sms);
  *used_tiled = tg.ok;
  if (tg.ok) {
    const TileInit<T> ti{nullptr, nullptr, nullptr, nullptr};
    rc = launch_tile<T, 1>(c, KC_SPMV, tg, true, a, ti, nullptr, nullptr, nullptr, c->cd_off);
    if (rc) return rc;
  } else {
    LAUNCH(c, KC_SPMV, (k_spmv<T, false>), c->grid_for((N + Vec<T>::W - 1) / Vec<T>::W), a, c->rs, (double*)nullptr,
           (const int*)nullptr, c->cd_off);
  }
  SIPB_CUDA_CHECK(cudaGetLastError());
  SIPB_CUDA_CHECK(cudaMemcpyAsync(y, dy.p, N * sizeof(T), cudaMemcpyDeviceToHost, c->stream));
  SIPB_CUDA_CHECK(cudaStreamSynchronize(c->stream));
  return SIPB_OK;
}

// The SpMV kernels of the CG as the solver launches them (unit tests): the argument block of a problem that holds Q in
// class form (tab, uploaded like Q_tab and opted in by tile_prepare) or as CDS arrays (R), the tile geometry of
// finalize, and the MODE 1 (y = Q x, dot(x, y)) or MODE 2 (CG prologue) kernel, tiled or generic.
template <typename T>
static int tile_probe_impl(sipb_ctx* c, const int64_t* n, int nd, const int64_t* offs, const void* tab, const void* R,
                           const void* x, const void* b, int mode, int tiled, void* y, void* r, void* p, void* x_old,
                           double* sums, int* geom) {
  const i64 N = n[0] * n[1] * n[2];
  const double hh[3] = {1, 1, 1};
  Problem<T> PB(c, sizeof(T) == 4 ? SIPB_F32 : SIPB_F64, 3, n, hh, false, true);
  PB.q_offs.assign(offs, offs + nd);
  PB.q_classes = tab != nullptr;
  if (PB.q_classes) {
    SIPB_CUDA_CHECK(PB.Q_tab.alloc((size_t)kMaxClasses * nd));
    SIPB_CUDA_CHECK(cudaMemsetAsync(PB.Q_tab.p, 0, (size_t)kMaxClasses * nd * sizeof(T), c->stream));
    SIPB_CUDA_CHECK(cudaMemcpyAsync(PB.Q_tab.p, tab, (size_t)27 * nd * sizeof(T), cudaMemcpyHostToDevice, c->stream));
  } else {
    int rc = upload_cds<T>(c, N, nd, R, PB.ld, PB.Q);
    if (rc) return rc;
  }
  const TileGeom tg = plan_tile<T>(3, n, false, PB.q_offs, n[2], 0, false, false, c->num_sms);
  if (geom) {
    const int gv[8] = {tg.ok, tg.TJ, tg.JT, tg.KC, tg.NS, tg.grid, tg.gpl, tg.LPP};
    memcpy(geom, gv, sizeof(gv));
  }
  SIPB_REQUIRE(!tiled || tg.ok, SIPB_E_UNSUPPORTED, "the tiled SpMV does not handle this grid");
  SIPB_REQUIRE(!(tiled && mode == 2 && !PB.q_classes), SIPB_E_UNSUPPORTED, "the tiled CG prologue has a class-form body only");
  if (tiled && PB.q_classes) { int rc = tile_prepare<T>(tg); if (rc) return rc; }
  DevBuf<T> dx, dy, db, dr, dp, dxo;
  SIPB_CUDA_CHECK(dx.alloc((size_t)N));
  SIPB_CUDA_CHECK(cudaMemcpyAsync(dx.p, x, N * sizeof(T), cudaMemcpyHostToDevice, c->stream));
  const i64 nvecN = (N + Vec<T>::W - 1) / Vec<T>::W;
  if (mode == 1) {
    SIPB_CUDA_CHECK(dy.alloc((size_t)N));
    const SpmvArgs<T> a = PB.spmv_args(dx.p, dy.p);
    if (tiled) {
      const TileInit<T> ti{nullptr, nullptr, nullptr, nullptr};
      int rc = launch_tile<T, 1>(c, KC_SPMV_DOT, tg, !PB.q_classes, a, ti, c->d_scal, nullptr, nullptr, c->cd_off);
      if (rc) return rc;
    } else {
      LAUNCH(c, KC_SPMV_DOT, (k_spmv<T, true>), c->grid_fit((const void*)k_spmv<T, true>, nvecN), a, c->rs, c->d_scal,
             (const int*)nullptr, c->cd_off);
    }
    SIPB_CUDA_CHECK(cudaGetLastError());
    SIPB_CUDA_CHECK(cudaMemcpyAsync(y, dy.p, N * sizeof(T), cudaMemcpyDeviceToHost, c->stream));
    SIPB_CUDA_CHECK(cudaMemcpyAsync(sums, c->d_scal, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    SIPB_CUDA_CHECK(cudaMemsetAsync(c->d_scal, 0, sizeof(double), c->stream));
  } else {
    SIPB_CUDA_CHECK(db.alloc((size_t)N));
    SIPB_CUDA_CHECK(dr.alloc((size_t)N));
    SIPB_CUDA_CHECK(dp.alloc((size_t)N));
    SIPB_CUDA_CHECK(dxo.alloc((size_t)N));
    SIPB_CUDA_CHECK(cudaMemcpyAsync(db.p, b, N * sizeof(T), cudaMemcpyHostToDevice, c->stream));
    const SpmvArgs<T> a = PB.spmv_args(dx.p, nullptr);
    if (tiled) {
      const TileInit<T> ti{db.p, dr.p, dp.p, dxo.p};
      int rc = launch_tile<T, 2>(c, KC_CG_INIT, tg, false, a, ti, nullptr, nullptr, c->d_cg, c->cd_off);
      if (rc) return rc;
    } else {
      LAUNCH(c, KC_CG_INIT, k_cg_init<T>, c->grid_for(nvecN), a, (const T*)db.p, dr.p, dp.p, dxo.p, c->rs, c->d_cg, c->cd_off);
    }
    SIPB_CUDA_CHECK(cudaGetLastError());
    SIPB_CUDA_CHECK(cudaMemcpyAsync(r, dr.p, N * sizeof(T), cudaMemcpyDeviceToHost, c->stream));
    SIPB_CUDA_CHECK(cudaMemcpyAsync(p, dp.p, N * sizeof(T), cudaMemcpyDeviceToHost, c->stream));
    SIPB_CUDA_CHECK(cudaMemcpyAsync(x_old, dxo.p, N * sizeof(T), cudaMemcpyDeviceToHost, c->stream));
    SIPB_CUDA_CHECK(cudaMemcpyAsync(sums, &c->d_cg->bb, 2 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));   // bb, rr
  }
  SIPB_CUDA_CHECK(cudaStreamSynchronize(c->stream));
  return SIPB_OK;
}

// The single-GPU cardinality select (unit tests), on a one-set problem with the identity operator, l = 0 and
// rho = gamma = 1, so that pass 1 of the y/l update produces v itself.  path 0 / 1: the sequence of the PARSDMM loop
// with the speculative levels off / on (pass 1, projector_params with deferred ties, pass 2); path 2: the sipb_project
// sequence (ties zeroed in place, then the apply pass).
template <typename T>
static int select_probe_impl(sipb_ctx* c, int64_t M, const void* v, int64_t k, uint64_t guess, int path, void* y,
                             int64_t* stats) {
  const int64_t nn[3] = {M, 1, 1};
  const double hh[3] = {1, 1, 1};
  Problem<T> P(c, sizeof(T) == 4 ? SIPB_F32 : SIPB_F64, 2, nn, hh, false, true);
  SetT<T> S;
  memset(&S.desc, 0, sizeof(S.desc));
  S.desc.set_kind = SIPB_SET_CARDINALITY;
  S.desc.op_kind = SIPB_OP_IDENTITY;
  S.desc.k = k;
  S.M = M;
  S.Mglob = M;
  S.op = identity_over(M);
  DevBuf<T> dv;
  SIPB_CUDA_CHECK(dv.alloc((size_t)M));
  SIPB_CUDA_CHECK(S.y.alloc((size_t)M));
  SIPB_CUDA_CHECK(S.l.alloc((size_t)M));
  SIPB_CUDA_CHECK(S.y_old.alloc((size_t)M));
  SIPB_CUDA_CHECK(S.s.alloc((size_t)M));
  SIPB_CUDA_CHECK(S.pp_y.alloc(1));
  SIPB_CUDA_CHECK(S.warm.alloc(2));
  SIPB_CUDA_CHECK(cudaMemcpyAsync(dv.p, v, M * sizeof(T), cudaMemcpyHostToDevice, c->stream));
  SIPB_CUDA_CHECK(cudaMemsetAsync(S.l.p, 0, M * sizeof(T), c->stream));
  SIPB_CUDA_CHECK(cudaMemsetAsync(S.y_old.p, 0, M * sizeof(T), c->stream));
  SIPB_CUDA_CHECK(cudaMemsetAsync(S.warm.p, 0, 2 * sizeof(double), c->stream));
  SIPB_CUDA_CHECK(cudaMemsetAsync(S.pp_y.p, 0, sizeof(ProjParams<T>), c->stream));
  const unsigned long long g64 = guess;
  SIPB_CUDA_CHECK(cudaMemcpyAsync(&S.pp_y.p->key_thr, &g64, sizeof(g64), cudaMemcpyHostToDevice, c->stream));
  const int slot = 10;
  i64 tie_chunk = 0;
  if (path == 2) {
    // project_impl: statistics, parameters with ties zeroed in place, the apply pass
    SIPB_CUDA_CHECK(cudaMemcpyAsync(S.y.p, dv.p, M * sizeof(T), cudaMemcpyDeviceToDevice, c->stream));
    LAUNCH(c, KC_VEC_STATS, k_vec_stats<T>, c->grid_for(M), M, S.y.p, c->rs, c->d_scal + slot);
    int rc = P.projector_params(S, S.y.p, slot, S.pp_y.p, S.warm.p, true);
    if (rc) return rc;
    LAUNCH(c, KC_FEAS, k_feas_dyn<T>, c->grid_for(M), M, S.y.p, (const T*)nullptr, P.proj_static(S, (T)1),
           (const ProjParams<T>*)S.pp_y.p, 1, c->rs, c->d_scal);
  } else {
    // Problem::solve, y/l update of a vector-mode cardinality set on one GPU
    const bool spec = path == 1;
    YlArgs<T> ya;
    memset(&ya, 0, sizeof(ya));
    ya.op = S.op;
    ya.P = P.proj_static(S, (T)1);
    ya.x = dv.p; ya.y = S.y.p; ya.l = S.l.p; ya.y_old = S.y_old.p; ya.s = S.s.p;
    ya.rho = (T)1; ya.gamma = (T)1;
    const i64 nvecM = (M + Vec<T>::W - 1) / Vec<T>::W;
    if (spec)
      LAUNCH(c, KC_YL_PASS1, (k_yl_spec<T>), c->grid_fit((const void*)k_yl_spec<T>, nvecM), ya, c->rs, c->d_scal + slot,
             &c->d_sel->spec_above, c->d_sel->spec, (const ProjParams<T>*)S.pp_y.p);
    else
      LAUNCH(c, KC_YL_PASS1, (k_yl<T, 1, false>), c->grid_fit((const void*)k_yl<T, 1, false>, nvecM), ya, c->rs,
             c->d_scal + slot);
    int rc = P.projector_params(S, S.y.p, slot, S.pp_y.p, S.warm.p, true, spec, &tie_chunk);
    if (rc) return rc;
    ya.dyn = S.pp_y.p;
    if (tie_chunk > 0) { ya.P.tie_base = c->d_tie_base; ya.P.tie_chunk = tie_chunk; }
    LAUNCH(c, KC_YL_PASS2, (k_yl<T, 2, false>), c->grid_fit((const void*)k_yl<T, 2, false>, nvecM), ya, c->rs, c->d_scal);
  }
  SIPB_CUDA_CHECK(cudaGetLastError());
  SIPB_CUDA_CHECK(cudaMemcpyAsync(y, S.y.p, M * sizeof(T), cudaMemcpyDeviceToHost, c->stream));
  ProjParams<T> pp;
  int sel[2];
  SIPB_CUDA_CHECK(cudaMemcpyAsync(&pp, S.pp_y.p, sizeof(pp), cudaMemcpyDeviceToHost, c->stream));
  SIPB_CUDA_CHECK(cudaMemcpyAsync(&sel[0], &c->d_sel->levels_run, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  SIPB_CUDA_CHECK(cudaMemcpyAsync(&sel[1], &c->d_sel->table_valid, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  SIPB_CUDA_CHECK(cudaMemsetAsync(c->d_scal, 0, (slot + 3) * sizeof(double), c->stream));
  SIPB_CUDA_CHECK(cudaStreamSynchronize(c->stream));
  // the chunk k_tie_cross settled in place: the one the quota boundary falls into (from its prefix and the counts)
  const int g = c->max_grid();
  int64_t cross = -1;
  if (tie_chunk > 0 && pp.need_ties) {
    std::vector<unsigned long long> cnt(g), base(g);
    SIPB_CUDA_CHECK(cudaMemcpy(cnt.data(), c->d_tie_counts, g * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    SIPB_CUDA_CHECK(cudaMemcpy(base.data(), c->d_tie_base, g * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    for (int q = 0; q < g; ++q)
      if (base[q] < pp.quota && base[q] + cnt[q] > pp.quota) cross = q;
  }
  if (stats) {
    const i64 chunk = ((M + g - 1) / g + kThreads - 1) / kThreads * kThreads;     // the row partition of the tie kernels
    const int64_t st[8] = {(int64_t)pp.key_thr, (int64_t)pp.quota, (int64_t)pp.count_eq, pp.need_ties, sel[0], sel[1],
                           (int64_t)chunk, cross};
    memcpy(stats, st, sizeof(st));
  }
  return SIPB_OK;
}

// One PARSDMM iteration's vector phases on a finalized single-GPU problem (unit tests): the caller's state is uploaded
// as the loop would leave it before iteration `it` (x stands for the CG's result), then rhs_phase and yl_phase run
// with the flags solve derives for that iteration.  Overwrites the problem's device vectors.
template <typename T>
static int iter_probe_impl(Problem<T>* P, int it, int do_adapt, const void* m_h, const void* x_h, const void* x_old_h,
                           const double* rho_d, const double* gamma_d, void* const* l_h, void* const* y_h,
                           void* const* y_prev_h, void* const* snap_h, const int* l1_inactive_prev, const double* warm,
                           const uint64_t* key_thr, void* rhs_h, void* const* s_h, double* slots, double* params,
                           int64_t* iparams, int64_t* launches, int* info) {
  sipb_ctx* c = P->ctx;
  const int p = (int)P->sets.size();
  const i64 N = P->N, npts = P->npts;
  c->reset_accounting();
  c->profile = false;
  std::vector<T> rho(p), gamma(p);
  for (int s = 0; s < p; ++s) { rho[s] = (T)rho_d[s]; gamma[s] = (T)gamma_d[s]; }
  auto up = [&](T* d, const void* h, i64 n) { return cudaMemcpyAsync(d, h, n * sizeof(T), cudaMemcpyHostToDevice, c->stream); };
  auto down = [&](void* h, const T* d, i64 n) { return cudaMemcpyAsync(h, d, n * sizeof(T), cudaMemcpyDeviceToHost, c->stream); };
  // m as solve uploads it ([m; 0] for Minkowski); the resident copy no longer belongs to a solve
  SIPB_CUDA_CHECK(up(P->m.p, m_h, npts));
  if (P->minkowski) SIPB_CUDA_CHECK(cudaMemsetAsync(P->m.p + npts, 0, npts * sizeof(T), c->stream));
  P->m_resident = false;
  SIPB_CUDA_CHECK(up(P->x.p, x_h, N));
  SIPB_CUDA_CHECK(up(P->x_old.p, x_old_h, N));
  SIPB_CUDA_CHECK(cudaMemsetAsync(c->d_scal, 0, kScalSlots * sizeof(double), c->stream));
  SIPB_CUDA_CHECK(cudaMemsetAsync(c->d_l1, 0, sizeof(L1State), c->stream));
  bool any_sparse = false;
  for (int s = 0; s < p; ++s) {
    SetT<T>& S = *P->sets[s];
    any_sparse = any_sparse || S.is_sparse;
    SIPB_CUDA_CHECK(up(S.l.p, l_h[s], S.M));
    SIPB_CUDA_CHECK(up(S.y.p, y_h[s], S.M));
    SIPB_CUDA_CHECK(up(S.y_old.p, y_prev_h[s], S.M));
    T* snaps[4] = {S.lhat0.p, S.s0.p, S.l0.p, S.y0.p};
    for (int q = 0; q < 4; ++q) SIPB_CUDA_CHECK(up(snaps[q], snap_h[4 * s + q], S.M));
    if (S.s.p) SIPB_CUDA_CHECK(cudaMemsetAsync(S.s.p, 0, S.M * sizeof(T), c->stream));
    SIPB_CUDA_CHECK(cudaMemcpyAsync(S.warm.p, warm + 2 * s, 2 * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    const unsigned long long k64 = key_thr[s];
    SIPB_CUDA_CHECK(cudaMemcpyAsync(&S.pp_y.p->key_thr, &k64, sizeof(k64), cudaMemcpyHostToDevice, c->stream));
    S.l1_inactive_prev = l1_inactive_prev[s] != 0;
  }
  SIPB_CUDA_CHECK(cudaStreamSynchronize(c->stream));   // the host staging above is pageable / on the stack
  // the flags of Problem::solve at iteration `it`
  const bool fuse_stop = !P->feas_only && !P->minkowski && getenv("SIPB_FUSE_STOP_OFF") == nullptr;
  const bool fuse_rdual = p <= kRdualSets && !any_sparse;
  int rc = P->rhs_phase(it, rho, fuse_rdual);
  if (rc) return rc;
  rc = P->yl_phase(it, rho, gamma, do_adapt != 0, fuse_stop, fuse_rdual);
  if (rc) return rc;
  rc = ctx_sync_scalars(c, true);
  if (rc) return rc;
  SIPB_REQUIRE(!c->h_l1->failed, SIPB_E_STATE, "l1 threshold search did not converge");
  SIPB_CUDA_CHECK(down(rhs_h, P->rhs.p, N));
  std::vector<ProjParams<T>> pp(p);
  for (int s = 0; s < p; ++s) {
    SetT<T>& S = *P->sets[s];
    SIPB_CUDA_CHECK(down(l_h[s], S.l.p, S.M));
    SIPB_CUDA_CHECK(down(y_h[s], S.y.p, S.M));
    const T* snaps[4] = {S.lhat0.p, S.s0.p, S.l0.p, S.y0.p};
    for (int q = 0; q < 4; ++q) SIPB_CUDA_CHECK(down(snap_h[4 * s + q], snaps[q], S.M));
    if (s_h && s_h[s] && S.s.p) SIPB_CUDA_CHECK(down(s_h[s], S.s.p, S.M));
    SIPB_CUDA_CHECK(cudaMemcpyAsync(&pp[s], S.pp_y.p, sizeof(ProjParams<T>), cudaMemcpyDeviceToHost, c->stream));
  }
  SIPB_CUDA_CHECK(cudaStreamSynchronize(c->stream));
  memcpy(slots, c->h_scal, kScalSlots * sizeof(double));
  for (int s = 0; s < p; ++s) {
    const double dp[3] = {(double)pp[s].theta, (double)pp[s].scale, (double)pp[s].fill};
    const int64_t ip[6] = {(int64_t)pp[s].key_thr, (int64_t)pp[s].quota, (int64_t)pp[s].count_eq, pp[s].keep_all,
                           pp[s].keep_none, pp[s].need_ties};
    memcpy(params + 3 * s, dp, sizeof(dp));
    memcpy(iparams + 6 * s, ip, sizeof(ip));
  }
  for (int q = 0; q < SIPB_N_KERNEL_CLASSES; ++q) launches[q] = c->launches[q];
  // the r_dual slots: fused, the rhs gather of `it` reduced iteration it-1 into the global slots (none at it = 1);
  // unfused, k_rdual reduced iteration `it` into each set's slot 3
  info[0] = fuse_rdual ? 1 : 0;
  info[1] = fuse_rdual ? it - 1 : it;
  info[2] = fuse_stop ? 1 : 0;
  info[3] = kSlotPerSet;
  info[4] = kSlotGlobal;
  return SIPB_OK;
}

template <typename T>
static int bench_spmv_impl(sipb_ctx* c, int ndim, const int64_t* n, int warmup, int reps, int flush_l2, double* avg_ms,
                           int64_t* alg_bytes, int form, int tiled) {
  const i64 N = n[0] * n[1] * (ndim == 3 ? n[2] : 1);
  const i64 ld = (N + 63) / 64 * 64;
  std::vector<int64_t> offs;
  // Q_offsets of bounds/identity + TV + distance in the reference's order: [0, -n1n2, -n1, -1, 1, n1, n1n2]
  offs.push_back(0);
  if (ndim == 3) offs.push_back(-n[0] * n[1]);
  offs.push_back(-n[0]); offs.push_back(-1); offs.push_back(1); offs.push_back(n[0]);
  if (ndim == 3) offs.push_back(n[0] * n[1]);
  const int nd = (int)offs.size();
  DevBuf<T> dR, dx, dy, flush, dtab;
  if (form == 1) {
    // stencil-class form: one row per class, the matrix is not streamed
    std::vector<T> tab((size_t)kMaxClasses * nd, (T)0.25);
    SIPB_CUDA_CHECK(dtab.alloc(tab.size()));
    SIPB_CUDA_CHECK(cudaMemcpyAsync(dtab.p, tab.data(), tab.size() * sizeof(T), cudaMemcpyHostToDevice, c->stream));
    SIPB_CUDA_CHECK(cudaStreamSynchronize(c->stream));
  }
  SIPB_CUDA_CHECK(dR.alloc(form == 1 ? 64 : (size_t)ld * nd));
  SIPB_CUDA_CHECK(dx.alloc((size_t)N));
  SIPB_CUDA_CHECK(dy.alloc((size_t)N));
  const size_t flush_elems = (size_t)(256u << 20) / sizeof(T);
  if (flush_l2) SIPB_CUDA_CHECK(flush.alloc(flush_elems));
  if (form != 1) LAUNCH(c, KC_FILL, k_fill<T>, c->max_grid(), (i64)ld * nd, dR.p, (T)0.25);
  LAUNCH(c, KC_FILL, k_fill<T>, c->max_grid(), N, dx.p, (T)1.5);
  // the argument block of a throw-away problem gives the class-form constants of the generic kernel too
  Problem<T> PB(c, sizeof(T) == 4 ? SIPB_F32 : SIPB_F64, ndim, n, std::vector<double>{1, 1, 1}.data(), false, true);
  PB.q_offs = offs;
  PB.q_classes = form == 1;
  SpmvArgs<T> a = PB.spmv_args(dx.p, dy.p);
  a.R = dR.p; a.ld = ld;
  a.tab = form == 1 ? dtab.p : nullptr;
  TileGeom tg;
  memset(&tg, 0, sizeof(tg));
  if (tiled) tg = plan_tile<T>(ndim, n, false, offs, ndim == 3 ? n[2] : 1, 0, false, false, c->num_sms);
  SIPB_REQUIRE(!tiled || tg.ok, SIPB_E_UNSUPPORTED, "the tiled SpMV does not handle this grid");
  const int g = c->grid_fit((const void*)k_spmv<T, true>, (N + Vec<T>::W - 1) / Vec<T>::W);
  cudaEvent_t e0, e1;
  SIPB_CUDA_CHECK(cudaEventCreate(&e0));
  SIPB_CUDA_CHECK(cudaEventCreate(&e1));
  double total = 0.0;
  for (int it = 0; it < warmup + reps; ++it) {
    if (flush_l2) LAUNCH(c, KC_FILL, k_fill<T>, c->max_grid(), (i64)flush_elems, flush.p, (T)it);
    SIPB_CUDA_CHECK(cudaEventRecord(e0, c->stream));
    if (tg.ok) {
      const TileInit<T> ti{nullptr, nullptr, nullptr, nullptr};
      int rc = launch_tile<T, 1>(c, KC_SPMV_DOT, tg, form != 1, a, ti, c->d_scal, nullptr, nullptr, c->cd_off);
      if (rc) return rc;
    } else {
      LAUNCH(c, KC_SPMV_DOT, (k_spmv<T, true>), g, a, c->rs, c->d_scal, (const int*)nullptr, c->cd_off);
    }
    SIPB_CUDA_CHECK(cudaEventRecord(e1, c->stream));
    SIPB_CUDA_CHECK(cudaEventSynchronize(e1));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    if (it >= warmup) total += ms;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  SIPB_CUDA_CHECK(cudaGetLastError());
  SIPB_CUDA_CHECK(cudaMemsetAsync(c->d_scal, 0, sizeof(double), c->stream));
  SIPB_CUDA_CHECK(cudaStreamSynchronize(c->stream));
  *avg_ms = total / std::max(1, reps);
  *alg_bytes = (int64_t)((form == 1 ? 0 : nd) + 2) * N * (int64_t)sizeof(T);
  return SIPB_OK;
}

}  // namespace sipb

extern "C" {

#define DISPATCH(dtype, fn, ...)                                                  \
  do {                                                                            \
    if ((dtype) == SIPB_F32) return fn<float>(__VA_ARGS__);                       \
    if ((dtype) == SIPB_F64) return fn<double>(__VA_ARGS__);                      \
    set_error("dtype must be SIPB_F32 or SIPB_F64");                              \
    return SIPB_E_INVALID;                                                        \
  } while (0)

int sipb_cds_spmv(sipb_ctx* ctx, int dtype, int64_t N, int nd, const void* R, const int64_t* offsets, const void* x,
                  void* y) {
  SIPB_REQUIRE(ctx && R && offsets && x && y, SIPB_E_INVALID, "null argument");
  SIPB_REQUIRE(nd >= 1 && nd <= kMaxDiag, SIPB_E_UNSUPPORTED, "number of diagonals outside [1,32]");
  SIPB_CUDA_CHECK(cudaSetDevice(ctx->device));
  DISPATCH(dtype, cds_spmv_impl, ctx, N, nd, R, offsets, x, y);
}
int sipb_cds_cg(sipb_ctx* ctx, int dtype, int64_t N, int nd, const void* R, const int64_t* offsets, const void* b,
                void* x, double tol, int max_iter, int* flag, double* relres, int* iters) {
  SIPB_REQUIRE(ctx && R && offsets && b && x && flag && relres && iters, SIPB_E_INVALID, "null argument");
  SIPB_REQUIRE(nd >= 1 && nd <= kMaxDiag, SIPB_E_UNSUPPORTED, "number of diagonals outside [1,32]");
  SIPB_CUDA_CHECK(cudaSetDevice(ctx->device));
  DISPATCH(dtype, cds_cg_impl, ctx, N, nd, R, offsets, b, x, tol, max_iter, flag, relres, iters);
}
int sipb_project(sipb_ctx* ctx, int dtype, const sipb_set_desc* desc, int64_t M, void* v, const void* m_vec) {
  SIPB_REQUIRE(ctx && desc && v, SIPB_E_INVALID, "null argument");
  SIPB_REQUIRE(desc->set_kind >= SIPB_SET_BOUNDS_SCALAR && desc->set_kind <= SIPB_SET_KIND_MAX, SIPB_E_UNSUPPORTED,
               "set type is outside the device hot path");
  if (desc->set_kind == SIPB_SET_BOUNDS_FIBER || desc->set_kind == SIPB_SET_CARD_FIBER ||
      desc->set_kind == SIPB_SET_CARD_SLICE) {
    SIPB_REQUIRE(desc->fiber_axis >= 0 && desc->fiber_axis < 3 && desc->td_n[0] >= 1 && desc->td_n[1] >= 1 &&
                     desc->td_n[2] >= 1 && desc->td_n[0] * desc->td_n[1] * desc->td_n[2] == M,
                 SIPB_E_INVALID, "td_n / fiber_axis do not match the vector");
  }
  SIPB_CUDA_CHECK(cudaSetDevice(ctx->device));
  DISPATCH(dtype, project_impl, ctx, desc, M, v, m_vec);
}
int sipb_op_apply(sipb_ctx* ctx, int dtype, int ndim, const int64_t* n, const double* h, int op_kind, int block_mode,
                  int adjoint, const void* in, void* out) {
  SIPB_REQUIRE(ctx && n && h && in && out, SIPB_E_INVALID, "null argument");
  SIPB_CUDA_CHECK(cudaSetDevice(ctx->device));
  DISPATCH(dtype, op_apply_impl, ctx, ndim, n, h, op_kind, block_mode, adjoint, in, out);
}
int sipb_sparse_apply(sipb_ctx* ctx, int dtype, const sipb_sparse* A, int adjoint, const void* in, void* out) {
  SIPB_REQUIRE(ctx && A && in && out, SIPB_E_INVALID, "null argument");
  SIPB_CUDA_CHECK(cudaSetDevice(ctx->device));
  DISPATCH(dtype, sparse_apply_impl, ctx, A, adjoint, in, out);
}
int sipb_cds_scaled_add(sipb_ctx* ctx, int dtype, int64_t N, int nd_a, void* A, const int64_t* a_offsets, int nd_b,
                        const void* B, const int64_t* b_offsets, double alpha) {
  SIPB_REQUIRE(ctx && A && a_offsets && B && b_offsets, SIPB_E_INVALID, "null argument");
  SIPB_CUDA_CHECK(cudaSetDevice(ctx->device));
  DISPATCH(dtype, cds_scaled_add_impl, ctx, N, nd_a, A, a_offsets, nd_b, B, b_offsets, alpha);
}
int sipb_bench_spmv(sipb_ctx* ctx, int dtype, int ndim, const int64_t* n, int warmup, int reps, int flush_l2,
                    double* avg_ms, int64_t* algorithmic_bytes) {
  SIPB_REQUIRE(ctx && n && avg_ms && algorithmic_bytes, SIPB_E_INVALID, "null argument");
  SIPB_CUDA_CHECK(cudaSetDevice(ctx->device));
  DISPATCH(dtype, bench_spmv_impl, ctx, ndim, n, warmup, reps, flush_l2, avg_ms, algorithmic_bytes, 0, 0);
}
int sipb_bench_spmv2(sipb_ctx* ctx, int dtype, int ndim, const int64_t* n, int warmup, int reps, int flush_l2, int form,
                     int tiled, double* avg_ms, int64_t* algorithmic_bytes) {
  SIPB_REQUIRE(ctx && n && avg_ms && algorithmic_bytes, SIPB_E_INVALID, "null argument");
  SIPB_REQUIRE(form == 0 || form == 1, SIPB_E_INVALID, "form must be 0 (CDS arrays) or 1 (stencil classes)");
  SIPB_CUDA_CHECK(cudaSetDevice(ctx->device));
  DISPATCH(dtype, bench_spmv_impl, ctx, ndim, n, warmup, reps, flush_l2, avg_ms, algorithmic_bytes, form, tiled);
}
int sipb_cds_spmv_grid(sipb_ctx* ctx, int dtype, const int64_t* n, int nd, const void* R, const int64_t* offsets,
                       const void* x, void* y, int* used_tiled) {
  SIPB_REQUIRE(ctx && n && R && offsets && x && y && used_tiled, SIPB_E_INVALID, "null argument");
  SIPB_REQUIRE(nd >= 1 && nd <= kMaxDiag, SIPB_E_UNSUPPORTED, "number of diagonals outside [1,32]");
  SIPB_REQUIRE(n[0] >= 2 && n[1] >= 2 && n[2] >= 2, SIPB_E_INVALID, "grid dimensions must be >= 2");
  SIPB_CUDA_CHECK(cudaSetDevice(ctx->device));
  DISPATCH(dtype, cds_spmv_grid_impl, ctx, n, nd, R, offsets, x, y, used_tiled);
}
int sipb_tile_probe(sipb_ctx* ctx, int dtype, const int64_t* n, int nd, const int64_t* offsets, const void* tab,
                    const void* R, const void* x, const void* b, int mode, int tiled, void* y, void* r, void* p,
                    void* x_old, double* sums, int* geom) {
  SIPB_REQUIRE(ctx && n && offsets && x && sums, SIPB_E_INVALID, "null argument");
  SIPB_REQUIRE((tab != nullptr) != (R != nullptr), SIPB_E_INVALID, "pass either a class table or CDS arrays");
  SIPB_REQUIRE(mode == 1 ? y != nullptr : (mode == 2 && b && r && p && x_old), SIPB_E_INVALID,
               "mode 1 needs y; mode 2 needs b, r, p and x_old");
  SIPB_REQUIRE(nd >= 1 && nd <= kTileDiag, SIPB_E_UNSUPPORTED, "number of diagonals outside [1,8]");
  SIPB_REQUIRE(n[0] >= 2 && n[1] >= 2 && n[2] >= 2, SIPB_E_INVALID, "grid dimensions must be >= 2");
  SIPB_REQUIRE(ctx->world <= 1, SIPB_E_UNSUPPORTED, "the probe runs on a single-GPU context");
  SIPB_CUDA_CHECK(cudaSetDevice(ctx->device));
  DISPATCH(dtype, tile_probe_impl, ctx, n, nd, offsets, tab, R, x, b, mode, tiled, y, r, p, x_old, sums, geom);
}
int sipb_select_probe(sipb_ctx* ctx, int dtype, int64_t M, const void* v, int64_t k, uint64_t guess, int path, void* y,
                      int64_t* stats) {
  SIPB_REQUIRE(ctx && v && y, SIPB_E_INVALID, "null argument");
  SIPB_REQUIRE(M >= 1 && path >= 0 && path <= 2, SIPB_E_INVALID, "M >= 1 and path 0, 1 or 2");
  SIPB_REQUIRE(ctx->world <= 1, SIPB_E_UNSUPPORTED, "the probe runs on a single-GPU context");
  SIPB_CUDA_CHECK(cudaSetDevice(ctx->device));
  DISPATCH(dtype, select_probe_impl, ctx, M, v, k, guess, path, y, stats);
}
int sipb_iter_probe(sipb_problem* pb, int it, int do_adapt, const void* m, const void* x, const void* x_old,
                    const double* rho, const double* gamma, void* const* l, void* const* y, void* const* y_prev,
                    void* const* snapshots, const int* l1_inactive_prev, const double* warm, const uint64_t* key_thr,
                    void* rhs, void* const* s, double* slots, double* params, int64_t* iparams, int64_t* launches,
                    int* info) {
  SIPB_REQUIRE(pb && m && x && x_old && rho && gamma && l && y && y_prev && snapshots && l1_inactive_prev && warm &&
                   key_thr && rhs && slots && params && iparams && launches && info,
               SIPB_E_INVALID, "null argument");
  SIPB_REQUIRE(it >= 1, SIPB_E_INVALID, "it must be >= 1");
  SIPB_CUDA_CHECK(cudaSetDevice(pb->ctx->device));
  if (pb->dtype == SIPB_F32) {
    auto* P = dynamic_cast<Problem<float>*>(pb);
    SIPB_REQUIRE(P && P->finalized, SIPB_E_STATE, "problem not finalized");
    SIPB_REQUIRE(!P->sg.on, SIPB_E_UNSUPPORTED, "the probe runs on a single-GPU problem (no slabs)");
    return iter_probe_impl<float>(P, it, do_adapt, m, x, x_old, rho, gamma, l, y, y_prev, snapshots, l1_inactive_prev,
                                  warm, key_thr, rhs, s, slots, params, iparams, launches, info);
  }
  auto* P = dynamic_cast<Problem<double>*>(pb);
  SIPB_REQUIRE(P && P->finalized, SIPB_E_STATE, "problem not finalized");
  SIPB_REQUIRE(!P->sg.on, SIPB_E_UNSUPPORTED, "the probe runs on a single-GPU problem (no slabs)");
  return iter_probe_impl<double>(P, it, do_adapt, m, x, x_old, rho, gamma, l, y, y_prev, snapshots, l1_inactive_prev,
                                 warm, key_thr, rhs, s, slots, params, iparams, launches, info);
}

}  // extern "C"
