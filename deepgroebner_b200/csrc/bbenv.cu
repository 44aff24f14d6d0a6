// bbenv.cu -- the extern "C" ABI (include/bbenv.h) of libbbenv.so: handle, arenas, host views, and dispatch to the
// per-NV kernel tables (bb_kernels.cuh, compiled in bb_nv.cu once per number of variables).  sm_100a only.
#include <cuda_runtime.h>
#include <emmintrin.h>

#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "bb_kernels.cuh"

// ------------------------------------------------------------------------------------------------ layout-free kernels
__global__ void __launch_bounds__(BB_THREADS) k_seed(BBParams P, const int* seeds, int base, int selection) {
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= P.num_envs) return;
  const uint32_t x = rng_seed(seeds ? seeds[e] : base + e);
  if (selection) P.st[e].sel_rng = x;
  else {
    P.st[e].rng = x;
    if (P.pre) { P.pre->count[e] = 0; P.pre->head[e] = 0; P.pre->rng[e] = x; }   // episodes prepared from the old stream are dropped
  }
}

// (re)starts the prefetch queues from every environment's current stream position / drops the queue of one environment
__global__ void __launch_bounds__(BB_THREADS) k_pre_flush(BBParams P, int only_env) {
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= P.num_envs || (only_env >= 0 && e != only_env)) return;
  P.pre->count[e] = 0; P.pre->head[e] = 0; P.pre->rng[e] = (uint32_t)P.st[e].rng;
}

__global__ void __launch_bounds__(BB_THREADS) k_fill_double(double* p, int n, double v) {
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e < n) p[e] = v;
}

// inverse table: every lane of a warp takes one residue; a^(p-2) by square and multiply
__global__ void __launch_bounds__(BB_THREADS) k_invtab(BBField F, uint16_t* tab) {
  uint32_t a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a < F.p) tab[a] = a ? (uint16_t)bbf_invmod(F, a) : 0;
}

__global__ void __launch_bounds__(BB_THREADS) k_pairs(BBParams P, int32_t* __restrict__ out,
                                                      int32_t* __restrict__ lengths, int pmax) {
  const int slot = (blockIdx.x * BB_THREADS + threadIdx.x) >> 5;
  if (slot >= P.num_envs) return;
  const int nP = P.st[slot].nP;
  const uint32_t* pairs = SLOT_PTR(uint32_t, P, slot, o_pairs);
  int32_t* o = out + (size_t)slot * pmax * 2;
  for (int r = bb_lane(); r < pmax; r += 32) {
    int i = -1, j = -1;
    if (r < nP) { uint32_t pr = pairs[r]; i = pr & 0xffffu; j = pr >> 16; }
    o[2 * r] = i; o[2 * r + 1] = j;
  }
  if (lengths && bb_lane() == 0) lengths[slot] = nP;
}

__global__ void __launch_bounds__(BB_THREADS) k_status(BBParams P, int32_t* status, bb_episode_stats* stats) {
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= P.num_envs) return;
  const BBEnvState& S = P.st[e];
  if (status) status[e] = S.status;
  if (stats) {
    bb_episode_stats o;
    memset(&o, 0, sizeof o);
    o.steps = S.steps; o.additions = S.adds; o.zero_reductions = S.zero; o.nonzero_reductions = S.nonzero;
    o.nbasis = S.nG; o.nterms = S.nT; o.status = S.status; o.rerolls = S.rerolls;
    o.trace_hash = S.trace_hash; o.discounted_return = S.disc_return;
    stats[e] = o;
  }
}

// Stream compaction of the environment list (north_star "batch management"): out[0] = number of RUNNING environments,
// out[1 ..] = every slot, RUNNING ones first, both groups in ascending order (a stable partition).  One CTA walks the
// status words in chunks of 1024: ballot + per-warp totals give each slot its rank inside the chunk.
__global__ void __launch_bounds__(1024) k_compact(BBParams P, int* __restrict__ out) {
  __shared__ int wsum[32];
  __shared__ int total;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int N = P.num_envs;
  int running = 0;
  for (int i = tid; i < N; i += 1024) running += P.st[i].status == BB_STATUS_RUNNING;
  running = __reduce_add_sync(0xffffffffu, running);
  if (lane == 0) wsum[wid] = running;
  __syncthreads();
  if (wid == 0) {
    const int t = __reduce_add_sync(0xffffffffu, wsum[lane]);
    if (lane == 0) { total = t; out[0] = t; }
  }
  __syncthreads();
  const int R = total;
  int before = 0;   // RUNNING environments in the chunks already placed
  for (int c0 = 0; c0 < N; c0 += 1024) {
    const int i = c0 + tid;
    const bool run = i < N && P.st[i].status == BB_STATUS_RUNNING;
    const unsigned m = __ballot_sync(0xffffffffu, run);
    __syncthreads();   // wsum of the previous chunk has been read
    if (lane == 0) wsum[wid] = __popc(m);
    __syncthreads();
    int wbefore = 0, chunk = 0;
    for (int w = 0; w < 32; w++) { const int v = wsum[w]; chunk += v; if (w < wid) wbefore += v; }
    const int rb = before + wbefore + __popc(m & ((1u << lane) - 1u));   // RUNNING environments before slot i
    if (i < N) out[1 + (run ? rb : R + i - rb)] = i;
    before += chunk;
  }
}

__global__ void __launch_bounds__(BB_THREADS) k_status_hist(BBParams P, int* __restrict__ hist) {
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= P.num_envs) return;
  const int st = P.st[e].status;
  atomicAdd(&hist[(unsigned)st < BB_STATUS_COUNT ? st : 0], 1);
}

// Discounted suffix sums inside episode segments (pg.discount_rewards, pg.py:18-39, on [N, T] trajectories):
// out[n][t] = x[n][t] + (done[n][t] ? 0 : gam * out[n][t+1]), one thread per trajectory walking backwards in fp64.
__global__ void __launch_bounds__(BB_THREADS) k_discount(int N, int T, const double* __restrict__ x,
                                                         const uint8_t* __restrict__ done, double gam, double* __restrict__ out) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  const double* xr = x + (size_t)n * T;
  const uint8_t* dr = done + (size_t)n * T;
  double* o = out + (size_t)n * T;
  double run = 0.0;
  for (int t = T - 1; t >= 0; t--) {
    run = dr[t] ? xr[t] : __dadd_rn(xr[t], __dmul_rn(gam, run));
    o[t] = run;
  }
}

// ------------------------------------------------------------------------------------------------ kernel tables
const BBKernelTable* bb_kernel_table_nv1(); const BBKernelTable* bb_kernel_table_nv2();
const BBKernelTable* bb_kernel_table_nv3(); const BBKernelTable* bb_kernel_table_nv4();
const BBKernelTable* bb_kernel_table_nv5(); const BBKernelTable* bb_kernel_table_nv6();
const BBKernelTable* bb_kernel_table_nv7(); const BBKernelTable* bb_kernel_table_nv8();

const BBKernelTable* bb_kernel_table(int nvars) {
  switch (nvars) {
    case 1: return bb_kernel_table_nv1(); case 2: return bb_kernel_table_nv2();
    case 3: return bb_kernel_table_nv3(); case 4: return bb_kernel_table_nv4();
    case 5: return bb_kernel_table_nv5(); case 6: return bb_kernel_table_nv6();
    case 7: return bb_kernel_table_nv7(); case 8: return bb_kernel_table_nv8();
  }
  return nullptr;
}

// ------------------------------------------------------------------------------------------------ host side
#ifndef BB_STAGE_SETS
#define BB_STAGE_SETS 3   // 4 (preparation three batches ahead) was measured: two preparations at once crowd out the next runner's CTAs
#endif
#ifndef BB_BANKS
#define BB_BANKS 3
#endif
struct bb_handle {
  bb_config cfg;
  BBParams P;
  BBLayout L;               // host-side (runtime) copy of the packed-monomial layout
  const BBKernelTable* K;   // kernels compiled for cfg.nvars
  int sm_count;
  std::vector<void*> allocs;
  std::string err;
  int* d_queue;             // bb_value's task counter
  int* d_ok;
  // Staging of bb_run, a ring of THREE sets: one compact slot per episode of a batch, holding the state right after
  // reset(), plus the batch's queue words and longest-predicted-first order.  While the runner works through one set
  // the next batches are prepared into the others on another stream (bb_prepare, or bb_run's own side stream when a
  // call spans several batches); three sets let the preparation run TWO batches ahead, which is what a pipeline
  // needs whose runners overlap (batch i + 1 starts in the tail of batch i, bb_run on alternating streams).
  struct Stage {
    int cap;                        // episodes it can hold (0 = not allocated yet)
    std::vector<void*> allocs;
    unsigned char* arena; BBEnvState* st;
    uint64_t* in_key; uint32_t* in_coef; int* in_off; int* in_np;
    int* order; uint8_t* cost_key;  // longest-predicted-first queue order of the batch (k_order)
    int* queue;                     // [BB_LPT_HIST + 2 * BB_LPT_BUCKETS] queue position, cost histogram, cursors
    cudaEvent_t prepared;           // recorded after k_prepare + k_order of the batch it holds
    cudaEvent_t consumed;           // recorded after the k_run that read it
    // the batch a bb_prepare call left here, waiting for its bb_run (episodes == 0: none)
    int episodes, seed_base; const int32_t* seeds;
    unsigned long long serial;      // order of the bb_prepare calls (the oldest matching batch is run first)
  } stage[BB_STAGE_SETS];
  unsigned long long stage_serial;
  int stage_next;                   // ring cursor: the set the next batch is prepared into (skipping waiting ones)
  cudaStream_t side;                // bb_run's own prepare stream (calls that span several batches)
  cudaEvent_t ev_entry;
  // bb_set_timing: events around the preparation and the runner of the LAST bb_run call (first batch)
  int timing; cudaEvent_t ev_t[3];
  // fork arena of bb_value: one full-size slot per worker warp
  int fork_cap;
  std::vector<void*> fork_allocs;
  unsigned char* fork_arena; BBEnvState* fork_st;
  // bb_step_host / bb_reset_host: pinned, device-mapped host staging (small batches: the kernel reads and writes it in
  // place) and a device twin (large batches: one async copy each way)
  unsigned char* host_stage; unsigned char* dev_stage; size_t stage_bytes;
  int sel_seed_stride;   // bb_run: episode e's Random-selection stream is seeded sel_seed_base + e * stride (default 1)
  int episode_offset;    // bb_run: global index of episode 0 of a call (bb_set_episode_offset: shards of one job)
  int nstaged;           // fixed ideals: environments 0 .. nstaged - 1 hold a staged ideal (bb_set_ideals)
  int* d_seeds; int* h_seeds; cudaEvent_t ev_seeds;   // bb_seed: device / pinned staging of explicit seeds
  // Environment arenas of bb_run: bank 0 is the handle's own (P: the environments of the step API); further banks, each a
  // full set of slots, are allocated the first time a bb_run call finds the earlier ones still in use by runners on other
  // streams.  With several banks the runners of consecutive batches overlap: the CTAs of batch i + 1 move in while batch i
  // drains (two streams fill the tail of a binomial batch; cyclic-6, whose launches last as long as their longest episode,
  // gains from a third).
  struct Bank {
    bool ready;
    unsigned char* arena; BBEnvState* st;
    uint64_t* gkey; uint32_t* gcoef; int* glen; int* gcount; uint64_t* grlm; uint32_t* gridx; uint32_t* gflag;
    int* queue;         // bb_reduce's query counter
    cudaEvent_t done;   // recorded after the last runner that used the bank
    cudaStream_t stream; // ... and the stream it ran on (calls on the same stream are ordered anyway)
    unsigned long long serial;   // order of use (all busy: queue behind the least recently taken)
  } bank[BB_BANKS];
  int* d_active;         // [num_envs + 1] slots of the RUNNING environments in ascending order, count in front (k_compact)
  int compaction;        // bb_set_compaction
  unsigned ticket;       // bb_step_host: sequence number the single-CTA kernel publishes in mapped host memory
  // prefetch queues of the step API (BBPre, bb_kernels.cuh): allocated on first use when the ideals are binomial draws
  int pre_depth;         // bb_set_prefetch: queue depth (0: off)
  bool pre_ready;
  BBPre* d_pre; BBParams preS; std::vector<void*> pre_allocs;
  // single-environment server (k_serve): bb_step_host / bb_reset_host / bb_observe_host of a one-environment handle talk to a
  // resident warp through a mailbox in mapped pinned memory instead of launching a kernel per call
  int serve_on;          // bb_set_serve (default: on when num_envs == 1)
  bool serving;          // an instance was launched and not yet joined
  BBMailbox* mb; size_t mb_bytes;
  unsigned serve_seq;
  cudaStream_t serve_stream; cudaEvent_t ev_serve;
  int prepare_by_warp;   // bb_run: 1 = episode preparation by one warp per episode even where the thread-per-episode kernel applies
  int two_term;    // bb_run: 1 = the two-term runner for binomial distributions (default), 0 = always the general one
  int run_wave[2];  // resident warps of the general (0) and the two-term (1) k_run on the device: the most either launches
  int policy_wave[4];  // resident warps of k_run_policy for hidden 32, 64, 128, 256 (0: not asked yet)
  int wide_mode;   // bb_run: reduce() by streams (k_run_wide): -1 = when the capacities ask for long polynomials, 0 = never, 1 = always, 2 / 3 / 7 / 8 = always, test configurations (bb_set_wide); 4 / 5 / 6 = 1 / 2 / 3
  // host mirrors of the distribution tables
  std::vector<double> cp;
  std::vector<char> staged;   // bb_set_ideals: which environments hold a staged ideal
};

static thread_local std::string g_create_err;

static int fail(bb_handle* h, const std::string& msg, int code = -1) {
  if (h) h->err = msg; else g_create_err = msg;
  return code;
}
#define CK(call)                                                                                      \
  do {                                                                                                \
    cudaError_t _e = (call);                                                                          \
    if (_e != cudaSuccess)                                                                            \
      return fail(h, std::string(#call) + ": " + cudaGetErrorString(_e), -2);                         \
  } while (0)

template <class T>
static cudaError_t dev_alloc(bb_handle* h, T** p, size_t count) {
  void* q = nullptr;
  cudaError_t e = cudaMalloc(&q, count * sizeof(T) + 16);
  if (e != cudaSuccess) return e;
  h->allocs.push_back(q);
  *p = (T*)q;
  return cudaMemset(q, 0, count * sizeof(T) + 16);
}

// One contiguous arena per slot from the capacities in P: 8-byte arrays first, every array 32-byte aligned, stride a
// multiple of 128.  Returns false if a slot would exceed 2 GiB.  hkey lies directly behind tkey and hcoef directly behind
// tcoef (max_terms is a multiple of 8, so no padding): scratch term i is term max_terms + i of the arena (bb_wide.cuh).
static bool layout_arena(BBParams& P) {
  size_t o = 0;
  auto take = [&o](size_t bytes) { size_t at = o; o = (o + bytes + 31) & ~(size_t)31; return (unsigned)at; };
  P.o_ghead = take(sizeof(GHeadMem) * (size_t)P.max_basis);
  P.o_lm = take(8 * (size_t)P.max_basis);
  P.o_rlm = take(8 * (size_t)P.max_basis);
  P.o_lscr = take(8 * (size_t)P.max_basis);
  P.o_plcm = take(8 * (size_t)P.max_pairs);
  P.o_tkey = take(8 * (size_t)P.max_terms);
  P.o_hkey = take(8 * 2 * (size_t)P.max_poly_terms);
  P.o_ridx = take(4 * (size_t)P.max_basis);
  P.o_pairs = take(4 * (size_t)P.max_pairs);
  P.o_tcoef = take(4 * (size_t)P.max_terms);
  P.o_hcoef = take(4 * 2 * (size_t)P.max_poly_terms);
  P.o_logit = take(4 * (size_t)P.max_pairs);
  if (o >= ((size_t)1 << 31)) return false;
  P.slot_stride = (o + 127) & ~(size_t)127;
  return true;
}

static inline int grid_for_warps_host(int nwarps) { return (nwarps + BB_WARPS - 1) / BB_WARPS; }

// ------------------------------------------------------------------------------------------------ single-environment server
#define BB_SERVE_IDLE_NS 10000000ull   // the resident warp leaves after 10 ms without a command

static inline void serve_post(bb_handle* h, unsigned cmd, int arg, int pmax, int pad) {
  // the whole command in one aligned 16-byte store (the device reads it with one 16-byte load)
  const unsigned seq = ++h->serve_seq;
  const __m128i w = _mm_set_epi32((int)(((unsigned)pmax << 1) | (pad ? 1u : 0u)), arg, (int)cmd, (int)seq);
  __atomic_thread_fence(__ATOMIC_RELEASE);
  _mm_store_si128(reinterpret_cast<__m128i*>(h->mb), w);
}

// Joins the server: asks a live instance to leave, waits for the kernel.  Every entry point that touches the environments
// or the handle's parameters by other means calls this first (ENTER).
static int serve_stop(bb_handle* h) {
  if (!h->serving) return 0;
  if (h->mb->alive) {
    serve_post(h, BB_CMD_STOP, 0, 0, 0);
    for (long spin = 0; spin < 200000000L && h->mb->alive && h->mb->done_seq != h->serve_seq; spin++) __builtin_ia32_pause();
  }
  CK(cudaStreamSynchronize(h->serve_stream));
  h->serving = false;
  return 0;
}

static int serve_launch(bb_handle* h, cudaStream_t s) {
  // after everything the caller enqueued on its stream (a seed, a reset of other state ...)
  CK(cudaEventRecord(h->ev_serve, s));
  CK(cudaStreamWaitEvent(h->serve_stream, h->ev_serve, 0));
  h->mb->alive = 1u;
  __atomic_thread_fence(__ATOMIC_RELEASE);
  CK(h->K->serve(h->P, h->mb, BB_SERVE_IDLE_NS, h->serve_stream));
  h->serving = true;
  return 0;
}

// One command through the mailbox: posts it, (re)starts the resident warp if none is polling, waits for the answer.
static int serve_call(bb_handle* h, unsigned cmd, int action, double* reward_host, uint8_t* done_host, int32_t* obs_host,
                      int32_t* lengths_host, int pmax, int pad, cudaStream_t s) {
  const BBParams& P = h->P;
  const int rows = obs_host ? pmax : 0;
  const size_t need = sizeof(BBMailbox) + 4 * (size_t)rows * P.cols + 64;
  if (need > h->mb_bytes) {
    int rc = serve_stop(h);
    if (rc < 0) return rc;
    if (h->mb) cudaFreeHost(h->mb);
    h->mb = nullptr; h->mb_bytes = 0;
    CK(cudaHostAlloc((void**)&h->mb, need, cudaHostAllocMapped));
    memset(h->mb, 0, need);
    h->mb_bytes = need;
    h->serve_seq = 0u;
  }
  BBMailbox* mb = h->mb;
  if (!h->serving || !mb->alive) { int rc = serve_launch(h, s); if (rc < 0) return rc; }
  serve_post(h, cmd, action, rows, pad);
  const unsigned seq = h->serve_seq;
  bool ok = false;
  for (int attempt = 0; attempt < 64 && !ok; attempt++) {
    for (long spin = 0; spin < 4000000L; spin++) {
      if (mb->done_seq == seq) { ok = true; break; }
      if ((spin & 1023) == 1023 && !mb->alive) break;   // the instance left (idle) before it saw the command
      __builtin_ia32_pause();
    }
    if (ok || mb->done_seq == seq) { ok = true; break; }
    if (!mb->alive) { int rc = serve_launch(h, s); if (rc < 0) return rc; }   // a new instance takes the pending command
    else if (cudaStreamQuery(h->serve_stream) != cudaErrorNotReady) {      // the kernel is gone without an answer: a fault
      CK(cudaStreamSynchronize(h->serve_stream));
      return fail(h, "bb_step_host: the environment server stopped without answering");
    }
  }
  if (!ok) return fail(h, "bb_step_host: the environment server did not answer");
  __atomic_thread_fence(__ATOMIC_ACQUIRE);
  const int len = mb->length;
  if (lengths_host) lengths_host[0] = len;
  if (cmd == BB_CMD_STEP) {
    if (reward_host) reward_host[0] = mb->reward;
    if (done_host) done_host[0] = (uint8_t)mb->done;
  }
  if (obs_host) {
    const size_t rowb = 4 * (size_t)P.cols;
    memcpy(obs_host, reinterpret_cast<const unsigned char*>(mb + 1), (size_t)(pad ? pmax : std::min(len, pmax)) * rowb);
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------ prefetch queues
#define BB_PRE_DEPTH 8        // episodes prepared ahead per environment; the queues are topped up every 4 * depth step calls
#define BB_PRE_MIN_ENVS 64    // below this a reset inside a step is not worth a queue (and a one-environment handle is served)
static bool layout_arena(BBParams& P);

static void pre_drop(bb_handle* h) {
  for (void* p : h->pre_allocs) cudaFree(p);
  h->pre_allocs.clear();
  h->pre_ready = false; h->d_pre = nullptr; h->P.pre = nullptr;
}

// Allocates the queues on first use (binomial draws with at most BB_PREP_S generators: what k_prefill's code prepares).
static int pre_setup(bb_handle* h, cudaStream_t s) {
  const BBParams& P = h->P;
  const bool want = h->pre_depth > 0 && P.dist.enabled && P.dist.kind == 0 && P.dist.s <= BB_PREP_S;
  if (!want) { if (h->pre_ready) { CK(cudaDeviceSynchronize()); pre_drop(h); } return 0; }
  if (h->pre_ready) return 0;
  BBParams S = P;
  S.pre = nullptr;
  S.max_basis = P.max_gens;
  S.max_pairs = std::max(1, P.max_gens * (P.max_gens - 1) / 2);
  S.max_terms = P.max_gen_terms;
  S.max_poly_terms = 1;
  if (!layout_arena(S)) return fail(h, "prefetch: staging slot too large");
  const size_t n = (size_t)P.num_envs * h->pre_depth, N = (size_t)P.num_envs;
  auto alloc = [&](void** out, size_t bytes) {
    cudaError_t e = cudaMalloc(out, bytes + 16);
    if (e == cudaSuccess) { h->pre_allocs.push_back(*out); e = cudaMemset(*out, 0, bytes + 16); }
    return e;
  };
  BBPre Q;
  CK(alloc((void**)&S.arena, n * S.slot_stride));
  CK(alloc((void**)&S.st, n * sizeof(BBEnvState)));
  S.num_envs = (int)n;
  S.in_key = nullptr; S.in_coef = nullptr; S.in_off = nullptr; S.in_np = nullptr;   // the lane code keeps the ideal in registers
  CK(alloc((void**)&Q.count, N * sizeof(int)));
  CK(alloc((void**)&Q.head, N * sizeof(int)));
  CK(alloc((void**)&Q.rng, N * sizeof(unsigned)));
  CK(alloc((void**)&Q.calls, sizeof(int)));
  CK(alloc((void**)&h->d_pre, sizeof(BBPre)));
  Q.S = S; Q.depth = h->pre_depth;
  CK(cudaMemcpy(h->d_pre, &Q, sizeof Q, cudaMemcpyHostToDevice));
  CK(cudaDeviceSynchronize());
  h->preS = S;
  h->P.pre = h->d_pre;
  h->pre_ready = true;
  k_pre_flush<<<(P.num_envs + BB_THREADS - 1) / BB_THREADS, BB_THREADS, 0, s>>>(h->P, -1);
  CK(cudaGetLastError());
  return 0;
}

// Before a call that may reset environments: the queues exist, and k_prefill goes with the call.  `now`: it tops the queues
// up; else it does so on every (4 * depth)-th step call by the device's own count (an environment takes at most one episode
// per step call, and on the binomial distributions an episode lasts tens of steps: a queue of `depth` outlasts 4 * depth
// calls except for runs of very short episodes, which then reset through the generator).
static int pre_refill(bb_handle* h, cudaStream_t s, bool now) {
  int rc = pre_setup(h, s);
  if (rc < 0 || !h->pre_ready) return rc;
  CK(h->K->prefill(h->P, h->preS, now ? 0 : 4 * h->pre_depth, s));
  return 0;
}

#define ENTER(h)                                                                                      \
  do {                                                                                                \
    CK(cudaSetDevice((h)->cfg.device));                                                               \
    if ((h)->serving) { int _rc = serve_stop(h); if (_rc < 0) return _rc; }                           \
  } while (0)

extern "C" {

int bb_abi_version(void) { return BB_ABI_VERSION; }

const char* bb_last_error(const bb_handle* h) { return h ? h->err.c_str() : g_create_err.c_str(); }
int bb_cols(const bb_handle* h) { return h->P.cols; }
int bb_num_envs(const bb_handle* h) { return h->P.num_envs; }
int bb_sm_count(const bb_handle* h) { return h->sm_count; }
uint64_t bb_hash_item(uint64_t x, uint64_t pos) { return bb_hash_item_impl(x, pos); }

int bb_resident_envs(int device, int nvars) {
  int sms = 0;
  const BBKernelTable* K = bb_kernel_table(nvars);
  if (!K) return -1;
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) return -1;
  if (cudaSetDevice(device) != cudaSuccess) return -1;
  // the larger wave of the two warp runners: a handle of this many slots keeps either of them fully resident, and bb_run
  // launches the other with no more warps than its own wave
  const int w0 = K->run_warps_per_sm(0), w1 = K->run_warps_per_sm(1);
  if (w0 <= 0 || w1 <= 0) return -1;
  return sms * std::max(w0, w1);
}

void bb_destroy(bb_handle* h) {
  if (!h) return;
  cudaSetDevice(h->cfg.device);
  serve_stop(h);
  if (h->mb) cudaFreeHost(h->mb);
  if (h->serve_stream) cudaStreamDestroy(h->serve_stream);
  if (h->ev_serve) cudaEventDestroy(h->ev_serve);
  for (void* p : h->allocs) cudaFree(p);
  for (int b = 0; b < BB_STAGE_SETS; b++) {
    for (void* p : h->stage[b].allocs) cudaFree(p);
    if (h->stage[b].prepared) cudaEventDestroy(h->stage[b].prepared);
    if (h->stage[b].consumed) cudaEventDestroy(h->stage[b].consumed);
  }
  for (int b = 0; b < BB_BANKS; b++) if (h->bank[b].done) cudaEventDestroy(h->bank[b].done);
  if (h->side) cudaStreamDestroy(h->side);
  if (h->ev_entry) cudaEventDestroy(h->ev_entry);
  if (h->ev_seeds) cudaEventDestroy(h->ev_seeds);
  for (int t = 0; t < 3; t++) if (h->ev_t[t]) cudaEventDestroy(h->ev_t[t]);
  if (h->h_seeds) cudaFreeHost(h->h_seeds);
  for (void* p : h->fork_allocs) cudaFree(p);
  for (void* p : h->pre_allocs) cudaFree(p);
  if (h->host_stage) cudaFreeHost(h->host_stage);
  if (h->dev_stage) cudaFree(h->dev_stage);
  delete h;
}

int bb_create(const bb_config* cfg, bb_handle** out) {
  bb_handle* h = nullptr;
  if (!cfg || !out) return fail(h, "bb_create: null argument");
  if (cfg->abi_version != BB_ABI_VERSION) return fail(h, "bb_create: ABI version mismatch");
  if (cfg->nvars < 1 || cfg->nvars > 8) return fail(h, "bb_create: nvars must be in 1..8");
  if (cfg->prime < 3 || cfg->prime > 65535) return fail(h, "bb_create: prime must be in 3..65535");
  for (int q = 2; q * q <= cfg->prime; q++)
    if (cfg->prime % q == 0) return fail(h, "bb_create: prime is not prime");
  if (cfg->k < 1) return fail(h, "bb_create: k must be >= 1");
  if (cfg->num_envs < 1) return fail(h, "bb_create: num_envs must be >= 1");
  if (cfg->max_basis < 2 || cfg->max_basis > 65535) return fail(h, "bb_create: max_basis must be in 2..65535");
  if (cfg->max_pairs < 1 || cfg->max_pairs > 65536) return fail(h, "bb_create: max_pairs must be in 1..65536");
  if (cfg->max_terms < 2 || cfg->max_poly_terms < 1 || cfg->max_gens < 1 || cfg->max_gen_terms < 1)
    return fail(h, "bb_create: capacities must be positive");
  if (cfg->max_gens > cfg->max_basis) return fail(h, "bb_create: max_gens exceeds max_basis");
  if ((unsigned)cfg->elimination > 2u || (unsigned)cfg->rewards > 1u) return fail(h, "bb_create: bad enum value");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(h, "bb_create: no CUDA device available (this library has no CPU fallback)", -3);
  if (cfg->device < 0 || cfg->device >= ndev) return fail(h, "bb_create: bad device ordinal");
  h = new bb_handle();
  h->cfg = *cfg;
  h->d_queue = nullptr; h->d_ok = nullptr;
  for (int b = 0; b < BB_STAGE_SETS; b++) {
    bb_handle::Stage& T = h->stage[b];
    T.cap = 0; T.arena = nullptr; T.st = nullptr; T.in_key = nullptr; T.in_coef = nullptr; T.in_off = nullptr; T.in_np = nullptr;
    T.order = nullptr; T.cost_key = nullptr; T.queue = nullptr; T.prepared = nullptr; T.consumed = nullptr;
    T.episodes = 0; T.seed_base = 0; T.seeds = nullptr; T.serial = 0;
  }
  for (int b = 0; b < BB_BANKS; b++) {
    h->bank[b].ready = false; h->bank[b].done = nullptr; h->bank[b].stream = nullptr; h->bank[b].serial = 0; h->bank[b].queue = nullptr;
  }
  h->stage_next = 0; h->stage_serial = 0; h->side = nullptr; h->ev_entry = nullptr; h->timing = 0;
  h->ev_t[0] = h->ev_t[1] = h->ev_t[2] = nullptr;
  h->episode_offset = 0; h->nstaged = 0; h->d_seeds = nullptr; h->h_seeds = nullptr; h->ev_seeds = nullptr;
  h->d_active = nullptr; h->compaction = 1; h->ticket = 0u;
  h->pre_depth = cfg->num_envs >= BB_PRE_MIN_ENVS ? BB_PRE_DEPTH : 0; h->pre_ready = false; h->d_pre = nullptr;
  h->serve_on = cfg->num_envs == 1 ? 1 : 0; h->serving = false; h->mb = nullptr; h->mb_bytes = 0; h->serve_seq = 0u;
  h->serve_stream = nullptr; h->ev_serve = nullptr;
  h->fork_cap = 0; h->fork_arena = nullptr; h->fork_st = nullptr;
  h->wide_mode = -1;
  h->prepare_by_warp = 0;
  h->two_term = 1;
  for (int u = 0; u < 4; u++) h->policy_wave[u] = 0;
  h->host_stage = nullptr; h->dev_stage = nullptr; h->stage_bytes = 0;
  h->sel_seed_stride = 1;
  auto bail = [&](int code) { g_create_err = h->err; bb_destroy(h); return code; };
#define CKC(call)                                                                                     \
  do {                                                                                                \
    cudaError_t _e = (call);                                                                          \
    if (_e != cudaSuccess) { h->err = std::string(#call) + ": " + cudaGetErrorString(_e); return bail(-2); } \
  } while (0)
  CKC(cudaSetDevice(cfg->device));
  cudaDeviceProp prop;
  CKC(cudaGetDeviceProperties(&prop, cfg->device));
  h->sm_count = prop.multiProcessorCount;
  BBParams& P = h->P;
  memset(&P, 0, sizeof P);
  h->L = bb_make_layout(cfg->nvars, (uint32_t)cfg->prime);
  h->K = bb_kernel_table(cfg->nvars);
  if (!h->K || h->K->w != h->L.w || h->K->dw != h->L.dw || h->K->dshift != h->L.dshift || h->K->eshift != h->L.eshift) {
    h->err = "bb_create: kernel table / layout mismatch"; return bail(-6);
  }
  for (int two = 0; two < 2; two++) {
    const int w = h->K->run_warps_per_sm(two);
    if (w <= 0) { h->err = "bb_create: k_run does not fit on the device"; return bail(-2); }
    h->run_wave[two] = w * h->sm_count;
  }
  P.F.p = h->L.p; P.F.mu = h->L.mu; P.nvars = cfg->nvars;
  P.num_envs = cfg->num_envs; P.k = cfg->k; P.cols = 2 * cfg->nvars * cfg->k;
  P.elimination = cfg->elimination; P.rewards = cfg->rewards;
  P.sort_input = cfg->sort_input ? 1 : 0; P.sort_reducers = cfg->sort_reducers ? 1 : 0;
  P.max_basis = cfg->max_basis; P.max_pairs = cfg->max_pairs; P.max_terms = (cfg->max_terms + 7) & ~7;
  P.max_poly_terms = cfg->max_poly_terms; P.max_gens = cfg->max_gens; P.max_gen_terms = cfg->max_gen_terms;
  P.obs_nv = cfg->nvars; P.max_episode_length = 0;
  const size_t N = (size_t)cfg->num_envs;
  if (!layout_arena(P)) { h->err = "bb_create: per-environment arena exceeds 2 GiB"; return bail(-1); }
  CKC(dev_alloc(h, &P.arena, N * P.slot_stride));
  CKC(dev_alloc(h, &P.st, N));
  CKC(dev_alloc(h, &P.in_key, N * P.max_gen_terms));
  CKC(dev_alloc(h, &P.in_coef, N * P.max_gen_terms));
  CKC(dev_alloc(h, &P.in_off, N * (P.max_gens + 1)));
  CKC(dev_alloc(h, &P.in_np, N));
  CKC(dev_alloc(h, &P.gkey, N * P.max_terms));
  CKC(dev_alloc(h, &P.gcoef, N * P.max_terms));
  CKC(dev_alloc(h, &P.glen, N * P.max_basis));
  CKC(dev_alloc(h, &P.gcount, N * 2));
  CKC(dev_alloc(h, &P.grlm, N * P.max_basis));
  CKC(dev_alloc(h, &P.gridx, N * P.max_basis));
  CKC(dev_alloc(h, &P.gflag, N * P.max_basis));
  CKC(dev_alloc(h, &P.counters, (size_t)CT_COUNT));
  {
    uint16_t* tab = nullptr;
    CKC(dev_alloc(h, &tab, (size_t)cfg->prime));
    k_invtab<<<(cfg->prime + BB_THREADS - 1) / BB_THREADS, BB_THREADS>>>(P.F, tab);
    CKC(cudaGetLastError());
    P.invtab = tab;
  }
  CKC(dev_alloc(h, &h->d_queue, (size_t)4));
  CKC(dev_alloc(h, &h->d_ok, (size_t)4));
  CKC(dev_alloc(h, &h->d_seeds, N));
  CKC(dev_alloc(h, &h->d_active, std::max(N + 1, (size_t)16)));
  for (int b = 0; b < BB_BANKS; b++) CKC(cudaEventCreateWithFlags(&h->bank[b].done, cudaEventDisableTiming));
  h->bank[0].ready = true;
  h->bank[0].arena = P.arena; h->bank[0].st = P.st; h->bank[0].gkey = P.gkey; h->bank[0].gcoef = P.gcoef; h->bank[0].glen = P.glen;
  h->bank[0].gcount = P.gcount; h->bank[0].grlm = P.grlm; h->bank[0].gridx = P.gridx; h->bank[0].gflag = P.gflag;
  CKC(dev_alloc(h, &h->bank[0].queue, (size_t)1));
  CKC(cudaHostAlloc((void**)&h->h_seeds, sizeof(int) * N, cudaHostAllocDefault));
  CKC(cudaEventCreateWithFlags(&h->ev_seeds, cudaEventDisableTiming));
  CKC(cudaEventCreateWithFlags(&h->ev_entry, cudaEventDisableTiming));
  CKC(cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking));
  CKC(cudaStreamCreateWithFlags(&h->serve_stream, cudaStreamNonBlocking));
  CKC(cudaEventCreateWithFlags(&h->ev_serve, cudaEventDisableTiming));
  for (int b = 0; b < BB_STAGE_SETS; b++) {
    CKC(dev_alloc(h, &h->stage[b].queue, (size_t)(BB_LPT_HIST + 2 * BB_LPT_BUCKETS)));
    CKC(cudaEventCreateWithFlags(&h->stage[b].prepared, cudaEventDisableTiming));
    CKC(cudaEventCreateWithFlags(&h->stage[b].consumed, cudaEventDisableTiming));
  }
  for (int t = 0; t < 3; t++) CKC(cudaEventCreate(&h->ev_t[t]));
  k_seed<<<(cfg->num_envs + BB_THREADS - 1) / BB_THREADS, BB_THREADS>>>(P, nullptr, 0, 0);
  k_seed<<<(cfg->num_envs + BB_THREADS - 1) / BB_THREADS, BB_THREADS>>>(P, nullptr, 0, 1);
  CKC(cudaGetLastError());
  CKC(cudaDeviceSynchronize());
#undef CKC
  *out = h;
  return 0;
}

// binomial(n,k) as ideals.cpp:67-72 computes it
static long long binom(int n, int k) {
  if (k < 0 || k > n) return 0;
  long long r = 1;
  for (int i = 1; i <= k; i++) r = r * (n - k + i) / i;
  return r;
}
// basis(n,d) order (ideals.cpp:39-64: permutations of d stars then n-1 bars == lex-descending exponent vectors)
static void basis_rec(const BBLayout& L, int n, int var, int left, int* e, std::vector<uint64_t>& out) {
  if (var == n - 1) { e[var] = left; out.push_back(bb_pack(L, e)); return; }
  for (int x = left; x >= 0; x--) { e[var] = x; basis_rec(L, n, var + 1, left - x, e, out); }
}

// kind 0: RandomBinomialIdealGenerator (ideals.cpp:157-201); kind 1: RandomIdealGenerator (ideals.cpp:204-231)
static int set_distribution_impl(bb_handle* h, int kind, int d, int s, double lam, int dist, int constants, int homogeneous,
                                 int pure) {
  if (!h) return -1;
  BBParams& P = h->P;
  if (d < 0 || s < 1) return fail(h, "bb_set_distribution: need d >= 0 and s >= 1");
  if (s > P.max_gens || 2 * s > P.max_gen_terms) return fail(h, "bb_set_distribution: s exceeds max_gens/max_gen_terms");
  if (kind == 1 && !(lam >= 0.0 && lam < 12.0))
    return fail(h, "bb_set_distribution_poly: lam must be in [0, 12) (libstdc++ switches to a rejection sampler at mean >= 12, "
                   "which is not restated on device)");
  if ((unsigned)dist > 2u) return fail(h, "bb_set_distribution: bad dist");
  if ((unsigned)d > h->L.emax || (unsigned)d > h->L.dmax) return fail(h, "bb_set_distribution: degree does not fit the packed layout");
  ENTER(h);
  const int n = h->L.n;
  // degree_distribution counts (ideals.cpp:75-100)
  std::vector<double> prob;
  prob.push_back(constants ? 1.0 : 0.0);
  if (dist == BB_DIST_UNIFORM) for (int i = 1; i <= d; i++) prob.push_back((double)binom(n + i - 1, n - 1));
  else if (dist == BB_DIST_WEIGHTED) for (int i = 0; i < d; i++) prob.push_back(1.0);
  else { for (int i = 0; i < d - 1; i++) prob.push_back(0.0); if (d >= 1) prob.push_back(1.0); }
  // std::discrete_distribution::param_type::_M_initialize (bits/random.tcc:2657-2678)
  std::vector<double> cp;
  if (prob.size() >= 2) {
    double sum = 0.0;
    for (double x : prob) sum += x;
    if (!(sum > 0.0)) return fail(h, "bb_set_distribution: empty degree distribution");
    for (double& x : prob) x /= sum;
    double acc = 0.0;
    for (size_t i = 0; i < prob.size(); i++) { acc = (i == 0) ? prob[0] : acc + prob[i]; cp.push_back(acc); }
    cp.back() = 1.0;
  }
  h->cp = cp;
  std::vector<uint64_t> basis; std::vector<int> off;
  for (int deg = 0; deg <= d; deg++) {
    off.push_back((int)basis.size());
    int e[8] = {0};
    basis_rec(h->L, n, 0, deg, e, basis);
  }
  off.push_back((int)basis.size());
  double* d_cp = nullptr; uint64_t* d_basis = nullptr; int* d_off = nullptr;
  CK(dev_alloc(h, &d_cp, cp.size() + 1));
  CK(dev_alloc(h, &d_basis, basis.size() + 1));
  CK(dev_alloc(h, &d_off, off.size()));
  if (!cp.empty()) CK(cudaMemcpy(d_cp, cp.data(), cp.size() * sizeof(double), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_basis, basis.data(), basis.size() * sizeof(uint64_t), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_off, off.data(), off.size() * sizeof(int), cudaMemcpyHostToDevice));
  if (h->pre_ready) { CK(cudaDeviceSynchronize()); pre_drop(h); }
  P.dist.enabled = 1; P.dist.d = d; P.dist.s = s; P.dist.homogeneous = homogeneous ? 1 : 0; P.dist.pure = pure ? 1 : 0;
  P.dist.ncp = (int)cp.size(); P.dist.cp = d_cp; P.dist.basis = d_basis; P.dist.basis_off = d_off;
  P.dist.kind = kind; P.dist.lm_thr = kind == 1 ? std::exp(-lam) : 0.0;
  return 0;
}

int bb_set_distribution(bb_handle* h, int d, int s, int dist, int constants, int homogeneous, int pure) {
  return set_distribution_impl(h, 0, d, s, 0.0, dist, constants, homogeneous, pure);
}
int bb_set_distribution_poly(bb_handle* h, int d, int s, double lam, int dist, int constants, int homogeneous) {
  return set_distribution_impl(h, 1, d, s, lam, dist, constants, homogeneous, 0);
}

// Seeds on `s`: explicit seeds travel through the handle's pinned staging (one async copy, no allocation, no device
// synchronisation; a second call waits for the first one's copy only if it is still in flight).
static int seed_impl(bb_handle* h, const int32_t* seeds, int base, int selection, cudaStream_t s) {
  if (!h) return -1;
  ENTER(h);
  const int* d_seeds = nullptr;
  if (seeds) {
    CK(cudaEventSynchronize(h->ev_seeds));
    memcpy(h->h_seeds, seeds, sizeof(int) * (size_t)h->P.num_envs);
    CK(cudaMemcpyAsync(h->d_seeds, h->h_seeds, sizeof(int) * (size_t)h->P.num_envs, cudaMemcpyHostToDevice, s));
    CK(cudaEventRecord(h->ev_seeds, s));
    d_seeds = h->d_seeds;
  }
  k_seed<<<(h->P.num_envs + BB_THREADS - 1) / BB_THREADS, BB_THREADS, 0, s>>>(h->P, d_seeds, base, selection);
  CK(cudaGetLastError());
  return 0;
}
int bb_seed(bb_handle* h, const int32_t* seeds, int base) { return seed_impl(h, seeds, base, 0, (cudaStream_t)0); }
int bb_seed_selection(bb_handle* h, const int32_t* seeds, int base) { return seed_impl(h, seeds, base, 1, (cudaStream_t)0); }
int bb_seed_on(bb_handle* h, const int32_t* seeds, int base, int selection, void* stream) {
  return seed_impl(h, seeds, base, selection ? 1 : 0, (cudaStream_t)stream);
}

int bb_set_ideals(bb_handle* h, const int32_t* env_ids, int count, const int32_t* ideal_offsets,
                  const int32_t* poly_offsets, const int32_t* exps, const int32_t* coefs) {
  if (!h) return -1;
  BBParams& P = h->P;
  if (count < 0 || !ideal_offsets || !poly_offsets || !exps || !coefs) return fail(h, "bb_set_ideals: null argument");
  ENTER(h);
  const int n = h->L.n;
  const BBLayout& L = h->L;
  std::vector<uint64_t> keys((size_t)P.max_gen_terms);
  std::vector<uint32_t> cf((size_t)P.max_gen_terms);
  std::vector<int> off((size_t)P.max_gens + 1);
  for (int c = 0; c < count; c++) {
    const int env = env_ids ? env_ids[c] : c;
    if (env < 0 || env >= P.num_envs) return fail(h, "bb_set_ideals: environment index out of range");
    const int p0 = ideal_offsets[c], p1 = ideal_offsets[c + 1];
    const int np = p1 - p0;
    if (np < 1 || np > P.max_gens) return fail(h, "bb_set_ideals: number of generators outside 1..max_gens");
    int nt = 0;
    off[0] = 0;
    for (int q = 0; q < np; q++) {
      const int t0 = poly_offsets[p0 + q], t1 = poly_offsets[p0 + q + 1];
      const int len = t1 - t0;
      if (len < 1) return fail(h, "bb_set_ideals: the zero polynomial is not a valid generator");
      if (nt + len > P.max_gen_terms) return fail(h, "bb_set_ideals: ideal exceeds max_gen_terms");
      std::vector<std::pair<uint64_t, uint32_t>> terms;
      for (int t = t0; t < t1; t++) {
        uint32_t deg = 0;
        for (int v = 0; v < n; v++) {
          int x = exps[(size_t)t * n + v];
          if (x < 0 || (uint32_t)x > L.emax) return fail(h, "bb_set_ideals: exponent does not fit the packed layout");
          deg += (uint32_t)x;
        }
        if (deg > L.dmax) return fail(h, "bb_set_ideals: degree does not fit the packed layout");
        long long cc = coefs[t] % (long long)L.p;
        if (cc < 0) cc += L.p;
        if (cc == 0) return fail(h, "bb_set_ideals: zero coefficient");
        terms.push_back({bb_pack(L, exps + (size_t)t * n), (uint32_t)cc});
      }
      std::stable_sort(terms.begin(), terms.end(), [](const auto& a, const auto& b) { return a.first < b.first; });
      for (size_t t = 1; t < terms.size(); t++)
        if (terms[t].first == terms[t - 1].first) return fail(h, "bb_set_ideals: repeated monomial in a generator");
      for (auto& tm : terms) { keys[nt] = tm.first; cf[nt] = tm.second; nt++; }
      off[q + 1] = nt;
    }
    CK(cudaMemcpy(P.in_key + (size_t)env * P.max_gen_terms, keys.data(), sizeof(uint64_t) * nt, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(P.in_coef + (size_t)env * P.max_gen_terms, cf.data(), sizeof(uint32_t) * nt, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(P.in_off + (size_t)env * (P.max_gens + 1), off.data(), sizeof(int) * (np + 1), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(P.in_np + env, &np, sizeof(int), cudaMemcpyHostToDevice));
    if (h->staged.empty()) h->staged.assign((size_t)P.num_envs, 0);
    h->staged[(size_t)env] = 1;
  }
  P.dist.enabled = 0;
  if (h->pre_ready) { CK(cudaDeviceSynchronize()); pre_drop(h); }
  // bb_run replays staged ideal (e mod nstaged): the staged environments must be a prefix 0 .. nstaged - 1
  h->nstaged = 0;
  while (h->nstaged < P.num_envs && !h->staged.empty() && h->staged[(size_t)h->nstaged]) h->nstaged++;
  return 0;
}

int bb_reset(bb_handle* h, const uint8_t* mask_dev, void* stream) {
  if (!h) return -1;
  ENTER(h);
  { int rc = pre_refill(h, (cudaStream_t)stream, true); if (rc < 0) return rc; }
  CK(h->K->reset(h->P, mask_dev, h->P.num_envs, (cudaStream_t)stream));
  return 0;
}

// Without auto-reset finished and faulted environments pile up over a batch of episodes: the step kernels then take the
// environments in RUNNING-first order (k_compact), so that the stepping warps sit in full CTAs.  With auto-reset every
// environment is RUNNING after every call and the list would be the identity.
static int compact_for_step(bb_handle* h, cudaStream_t s, const int** active) {
  *active = nullptr;
  if (!h->compaction || h->P.auto_reset || h->P.num_envs < 2 * BB_WARPS) return 0;
  k_compact<<<1, 1024, 0, s>>>(h->P, h->d_active);
  CK(cudaGetLastError());
  *active = h->d_active;
  return 0;
}

int bb_step(bb_handle* h, const int32_t* actions_dev, double* reward_dev, uint8_t* done_dev, void* stream) {
  if (!h) return -1;
  if (!actions_dev) return fail(h, "bb_step: null actions");
  ENTER(h);
  const int* active = nullptr;
  int rc = h->P.auto_reset ? pre_refill(h, (cudaStream_t)stream, false) : 0;
  if (rc < 0) return rc;
  rc = compact_for_step(h, (cudaStream_t)stream, &active);
  if (rc < 0) return rc;
  CK(h->K->step(h->P, actions_dev, reward_dev, done_dev, active, h->P.num_envs, (cudaStream_t)stream));
  return 0;
}

// ---- the reference binding's calls with HOST buffers (wrapped.pyx:18-26): one launch, one synchronisation
#define BB_ZERO_COPY_BYTES (256u << 10)
static int host_call(bb_handle* h, int do_step, const int32_t* actions_host, double* reward_host, uint8_t* done_host,
                     int32_t* obs_host, int32_t* lengths_host, int pmax, int pad, cudaStream_t s) {
  const BBParams& P = h->P;
  const size_t N = (size_t)P.num_envs;
  if (pmax < 0 || (obs_host && pmax < 1)) return fail(h, "bb_step_host / bb_reset_host: bad pmax");
  if (do_step == 1 && !actions_host) return fail(h, "bb_step_host: null actions");
  if (h->serve_on && P.num_envs == 1)   // one environment: a command to the resident warp instead of a launch
    return serve_call(h, do_step == 1 ? BB_CMD_STEP : (do_step == 2 ? BB_CMD_RESET : BB_CMD_OBSERVE), do_step == 1 ? actions_host[0] : 0,
                      reward_host, done_host, obs_host, lengths_host, pmax, pad, s);
  if (h->serving) { int rc = serve_stop(h); if (rc < 0) return rc; }
  if (do_step == 2 || (do_step == 1 && P.auto_reset)) { int rc = pre_refill(h, s, do_step == 2); if (rc < 0) return rc; }
  if (do_step == 2) { CK(h->K->reset(h->P, nullptr, P.num_envs, s)); do_step = 0; }
  // staging layout: reward f64[N] | obs i32[N * pmax * cols] | lengths i32[N] | actions i32[N] | done u8[N] | ticket u32
  const size_t o_rew = 0, o_obs = o_rew + 8 * N, o_len = o_obs + (obs_host ? 4 * N * (size_t)pmax * P.cols : 0);
  const size_t o_act = o_len + 4 * N, o_done = o_act + 4 * N, o_tick = (o_done + N + 15) & ~(size_t)15, bytes = o_tick + 16;
  if (bytes > h->stage_bytes) {
    CK(cudaStreamSynchronize(s));
    if (h->host_stage) cudaFreeHost(h->host_stage);
    if (h->dev_stage) cudaFree(h->dev_stage);
    h->host_stage = nullptr; h->dev_stage = nullptr; h->stage_bytes = 0;
    CK(cudaHostAlloc((void**)&h->host_stage, bytes, cudaHostAllocMapped));
    CK(cudaMalloc((void**)&h->dev_stage, bytes));
    h->stage_bytes = bytes;
  }
  const bool zero_copy = bytes <= BB_ZERO_COPY_BYTES;
  unsigned char* hs = h->host_stage;
  unsigned char* ds = zero_copy ? hs : h->dev_stage;   // UVA: mapped pinned memory is addressable from the device as it is
  const int* d_actions = nullptr;
  int action0 = 0;
  if (do_step) {
    if (N == 1) action0 = actions_host[0];   // by value in the launch parameters
    else {
      memcpy(hs + o_act, actions_host, 4 * N);
      if (!zero_copy) CK(cudaMemcpyAsync(ds + o_act, hs + o_act, 4 * N, cudaMemcpyHostToDevice, s));
      d_actions = (const int*)(ds + o_act);
    }
  }
  const int* active = nullptr;
  if (do_step) { int rc = compact_for_step(h, s, &active); if (rc < 0) return rc; }
  // one CTA writing mapped host memory: the host waits for the kernel's ticket in that memory (a few hundred nanoseconds
  // after the kernel's last store) instead of a stream synchronisation through the driver
  const bool poll = zero_copy && P.num_envs <= BB_WARPS && !active;
  volatile unsigned* tick = reinterpret_cast<volatile unsigned*>(hs + o_tick);
  const unsigned ticket = ++h->ticket ? h->ticket : ++h->ticket;   // never 0
  if (poll) *tick = 0u;
  CK(h->K->step_obs(P, d_actions, action0, do_step ? (double*)(ds + o_rew) : nullptr, do_step ? (uint8_t*)(ds + o_done) : nullptr,
                    obs_host ? (int32_t*)(ds + o_obs) : nullptr, (int32_t*)(ds + o_len), pmax, pad, do_step, active,
                    poll ? (unsigned*)(hs + o_tick) : nullptr, ticket, P.num_envs, s));
  if (!zero_copy) {
    CK(cudaMemcpyAsync(hs, ds, o_act, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(hs + o_done, ds + o_done, N, cudaMemcpyDeviceToHost, s));
  }
  bool seen = false;
  if (poll) {
    for (long spin = 0; spin < 4000000L; spin++) {   // ~ a few milliseconds, then the ordinary wait (which also reports faults)
      if (*tick == ticket) { seen = true; break; }
      __builtin_ia32_pause();
    }
  }
  if (!seen) CK(cudaStreamSynchronize(s));
  __atomic_thread_fence(__ATOMIC_ACQUIRE);   // the results below are read after the ticket
  const int32_t* len = (const int32_t*)(hs + o_len);
  if (lengths_host) memcpy(lengths_host, len, 4 * N);
  if (do_step && reward_host) memcpy(reward_host, hs + o_rew, 8 * N);
  if (do_step && done_host) memcpy(done_host, hs + o_done, N);
  if (obs_host) {
    const size_t rowb = 4 * (size_t)P.cols;
    if (pad) memcpy(obs_host, hs + o_obs, N * (size_t)pmax * rowb);
    else for (size_t e = 0; e < N; e++)
      memcpy(obs_host + e * (size_t)pmax * P.cols, hs + o_obs + e * (size_t)pmax * rowb, (size_t)std::min(len[e], pmax) * rowb);
  }
  return 0;
}

int bb_step_observe(bb_handle* h, const int32_t* actions_dev, double* reward_dev, uint8_t* done_dev, int32_t* obs_dev,
                    int32_t* lengths_dev, int pmax, void* stream) {
  if (!h) return -1;
  if (!actions_dev || pmax < 0 || (obs_dev && pmax < 1)) return fail(h, "bb_step_observe: bad argument");
  ENTER(h);
  const int* active = nullptr;
  int rc = h->P.auto_reset ? pre_refill(h, (cudaStream_t)stream, false) : 0;
  if (rc < 0) return rc;
  rc = compact_for_step(h, (cudaStream_t)stream, &active);
  if (rc < 0) return rc;
  CK(h->K->step_obs(h->P, actions_dev, 0, reward_dev, done_dev, obs_dev, lengths_dev, pmax, 1, 1, active, nullptr, 0u,
                    h->P.num_envs, (cudaStream_t)stream));
  return 0;
}

int bb_step_host(bb_handle* h, const int32_t* actions_host, double* reward_host, uint8_t* done_host, int32_t* obs_host,
                 int32_t* lengths_host, int pmax, int pad, void* stream) {
  if (!h) return -1;
  CK(cudaSetDevice(h->cfg.device));
  return host_call(h, 1, actions_host, reward_host, done_host, obs_host, lengths_host, pmax, pad, (cudaStream_t)stream);
}

int bb_reset_host(bb_handle* h, int32_t* obs_host, int32_t* lengths_host, int pmax, int pad, void* stream) {
  if (!h) return -1;
  CK(cudaSetDevice(h->cfg.device));
  return host_call(h, 2, nullptr, nullptr, nullptr, obs_host, lengths_host, pmax, pad, (cudaStream_t)stream);
}

int bb_observe_host(bb_handle* h, int32_t* obs_host, int32_t* lengths_host, int pmax, int pad, void* stream) {
  if (!h) return -1;
  CK(cudaSetDevice(h->cfg.device));
  return host_call(h, 0, nullptr, nullptr, nullptr, obs_host, lengths_host, pmax, pad, (cudaStream_t)stream);
}

int bb_select(bb_handle* h, int strategy, int32_t* actions_dev, void* stream) {
  if (!h) return -1;
  if ((unsigned)strategy > 8u || !actions_dev) return fail(h, "bb_select: bad argument");
  ENTER(h);
  CK(h->K->select(h->P, strategy, actions_dev, h->P.num_envs, (cudaStream_t)stream));
  return 0;
}

int bb_observe(bb_handle* h, int32_t* obs_dev, int32_t* lengths_dev, int pmax, void* stream) {
  if (!h) return -1;
  if (pmax < 0 || (obs_dev && pmax == 0)) return fail(h, "bb_observe: bad pmax");
  ENTER(h);
  CK(h->K->observe(h->P, obs_dev, lengths_dev, pmax, h->P.num_envs, (cudaStream_t)stream));
  return 0;
}

int bb_pairs(bb_handle* h, int32_t* pairs_dev, int32_t* lengths_dev, int pmax, void* stream) {
  if (!h) return -1;
  if (!pairs_dev || pmax < 1) return fail(h, "bb_pairs: bad argument");
  ENTER(h);
  k_pairs<<<grid_for_warps_host(h->P.num_envs), BB_THREADS, 0, (cudaStream_t)stream>>>(h->P, pairs_dev, lengths_dev, pmax);
  CK(cudaGetLastError());
  return 0;
}

int bb_status(bb_handle* h, int32_t* status_dev, void* stream) {
  if (!h) return -1;
  ENTER(h);
  k_status<<<(h->P.num_envs + BB_THREADS - 1) / BB_THREADS, BB_THREADS, 0, (cudaStream_t)stream>>>(h->P, status_dev, nullptr);
  CK(cudaGetLastError());
  return 0;
}

int bb_stats(bb_handle* h, bb_episode_stats* stats_dev, void* stream) {
  if (!h) return -1;
  ENTER(h);
  k_status<<<(h->P.num_envs + BB_THREADS - 1) / BB_THREADS, BB_THREADS, 0, (cudaStream_t)stream>>>(h->P, nullptr, stats_dev);
  CK(cudaGetLastError());
  return 0;
}

// Staging parameters for a batch in set `which`: a copy of P whose arena is the compact per-episode one (capacity: the
// input ideal only -- max_gens polynomials, all their pairs, max_gen_terms terms).
#define BB_RUN_BATCH 65536
static int stage_params(bb_handle* h, int which, int batch, BBParams& S) {
  const BBParams& P = h->P;
  bb_handle::Stage& T = h->stage[which];
  S = P;
  S.pre = nullptr;
  S.max_basis = P.max_gens;
  S.max_pairs = std::max(1, P.max_gens * (P.max_gens - 1) / 2);
  S.max_terms = P.max_gen_terms;
  S.max_poly_terms = 1;
  if (!layout_arena(S)) return fail(h, "bb_run: staging slot too large");
  if (batch > T.cap) {
    CK(cudaDeviceSynchronize());   // the set is about to be replaced (first call, or a larger batch than ever before)
    for (void* p : T.allocs) cudaFree(p);
    T.allocs.clear();
    T.cap = 0;
    const size_t n = (size_t)batch;
    auto alloc = [&](void** out, size_t bytes) {
      cudaError_t e = cudaMalloc(out, bytes + 16);
      if (e == cudaSuccess) { T.allocs.push_back(*out); e = cudaMemset(*out, 0, bytes + 16); }
      return e;
    };
    CK(alloc((void**)&T.arena, n * S.slot_stride));
    CK(alloc((void**)&T.st, n * sizeof(BBEnvState)));
    CK(alloc((void**)&T.in_key, n * P.max_gen_terms * sizeof(uint64_t)));
    CK(alloc((void**)&T.in_coef, n * P.max_gen_terms * sizeof(uint32_t)));
    CK(alloc((void**)&T.in_off, n * (P.max_gens + 1) * sizeof(int)));
    CK(alloc((void**)&T.in_np, n * sizeof(int)));
    CK(alloc((void**)&T.order, n * sizeof(int)));
    CK(alloc((void**)&T.cost_key, n));
    CK(cudaDeviceSynchronize());
    T.cap = batch;
  }
  S.arena = T.arena; S.st = T.st; S.num_envs = batch;
  if (P.dist.enabled) {  // generated ideals are staged per episode; fixed ideals are read in place from the handle
    S.in_key = T.in_key; S.in_coef = T.in_coef; S.in_off = T.in_off; S.in_np = T.in_np;
  }
  return 0;
}

// The part of BBRunArgs the preparation reads, for episodes [base, base + count) of a call
static void prepare_args(bb_handle* h, int which, int base, int count, int seed_base, const int32_t* seeds_dev, BBRunArgs& A) {
  memset(&A, 0, sizeof A);
  const bb_handle::Stage& T = h->stage[which];
  A.episodes = count; A.seed_base = seed_base; A.seeds = seeds_dev; A.ep_base = base;
  A.ep_offset = h->episode_offset; A.nstaged = std::max(1, h->nstaged);
  A.queue = T.queue; A.order = T.order; A.cost_key = T.cost_key; A.prepare_by_warp = h->prepare_by_warp;
}

// k_prepare + k_order of one batch into set `which` on stream ps; the set's previous reader must have finished.
static int enqueue_prepare(bb_handle* h, int which, int base, int count, int seed_base, const int32_t* seeds_dev, cudaStream_t ps) {
  BBParams S;
  int rc = stage_params(h, which, std::max(count, h->stage[which].cap), S);
  if (rc < 0) return rc;
  bb_handle::Stage& T = h->stage[which];
  BBRunArgs A;
  prepare_args(h, which, base, count, seed_base, seeds_dev, A);
  CK(cudaStreamWaitEvent(ps, T.consumed, 0));
  CK(cudaStreamWaitEvent(ps, T.prepared, 0));   // a bb_prepare whose batch was never run may still be writing the set
  CK(cudaMemsetAsync(T.queue, 0, sizeof(int) * (BB_LPT_HIST + 2 * BB_LPT_BUCKETS), ps));
  CK(h->K->prepare(S, A, ps));
  CK(cudaEventRecord(T.prepared, ps));
  return 0;
}

static int check_staged(bb_handle* h, const char* who) {
  if (!h->P.dist.enabled && h->nstaged < 1)
    return fail(h, std::string(who) + ": no ideal distribution set and no ideal staged in environment 0 (bb_set_ideals)");
  return 0;
}

// The next set of the ring that no prepared batch is waiting in (all waiting: the oldest one is given up).
static int stage_take(bb_handle* h) {
  int which = h->stage_next;
  for (int t = 0; t < BB_STAGE_SETS && h->stage[which].episodes != 0; t++) which = (which + 1) % BB_STAGE_SETS;
  h->stage[which].episodes = 0;
  h->stage_next = (which + 1) % BB_STAGE_SETS;
  return which;
}

int bb_prepare(bb_handle* h, int episodes, int seed_base, const int32_t* seeds_dev, void* stream) {
  if (!h) return -1;
  if (episodes < 1 || episodes > BB_RUN_BATCH) return fail(h, "bb_prepare: episodes must be in 1..65536 (one batch)");
  ENTER(h);
  int rc = check_staged(h, "bb_prepare");
  if (rc < 0) return rc;
  const int which = stage_take(h);
  rc = enqueue_prepare(h, which, 0, episodes, seed_base, seeds_dev, (cudaStream_t)stream);
  if (rc < 0) return rc;
  bb_handle::Stage& T = h->stage[which];
  T.episodes = episodes; T.seed_base = seed_base; T.seeds = seeds_dev; T.serial = ++h->stage_serial;
  return 0;
}

static int check_sink(bb_handle* h, const bb_poly_sink* k, const char* which, const char* fn = "bb_run_export") {
  if (!k) return 0;
  if (!k->lens_dev || !k->exps_dev || !k->coefs_dev || !k->where_dev || !k->used_dev)
    return fail(h, std::string(fn) + ": the " + which + " sink has a NULL buffer");
  if (k->cap_polys < 0 || k->cap_terms < 0)
    return fail(h, std::string(fn) + ": the " + which + " sink has a negative capacity");
  return 0;
}

// The environment bank of a bb_run / bb_reduce call on stream s: the one this stream used last (calls on a stream are ordered
// anyway), else the first bank no kernel on another stream may still be using (allocated on first use), else the least
// recently taken one, which s then waits for.  PB receives the handle's parameters on that bank; returns its index or < 0.
// The caller records the bank's `done` event after its last kernel.
static int take_bank(bb_handle* h, cudaStream_t s, BBParams& PB) {
  int bk = -1;
  for (int b = 0; b < BB_BANKS && bk < 0; b++)
    if (h->bank[b].ready && h->bank[b].stream == s) bk = b;
  if (bk < 0) {
    for (int b = 0; b < BB_BANKS && bk < 0; b++) {
      bb_handle::Bank& B = h->bank[b];
      if (!B.ready) {
        const size_t N = (size_t)h->P.num_envs;
        const BBParams& P = h->P;
        CK(dev_alloc(h, &B.arena, N * P.slot_stride));
        CK(dev_alloc(h, &B.st, N));
        CK(dev_alloc(h, &B.gkey, N * P.max_terms));
        CK(dev_alloc(h, &B.gcoef, N * P.max_terms));
        CK(dev_alloc(h, &B.glen, N * P.max_basis));
        CK(dev_alloc(h, &B.gcount, N * 2));
        CK(dev_alloc(h, &B.grlm, N * P.max_basis));
        CK(dev_alloc(h, &B.gridx, N * P.max_basis));
        CK(dev_alloc(h, &B.gflag, N * P.max_basis));
        CK(dev_alloc(h, &B.queue, (size_t)1));
        CK(cudaDeviceSynchronize());   // the allocations' memsets ran on the legacy stream
        B.ready = true;
        bk = b;
      } else if (cudaEventQuery(B.done) == cudaSuccess) {
        bk = b;
      } else {
        (void)cudaGetLastError();   // cudaErrorNotReady is not an error
      }
    }
    if (bk < 0) {   // every bank is in use elsewhere: queue behind the least recently taken
      bk = 0;
      for (int b = 1; b < BB_BANKS; b++) if (h->bank[b].serial < h->bank[bk].serial) bk = b;
      CK(cudaStreamWaitEvent(s, h->bank[bk].done, 0));
    }
  }
  h->bank[bk].stream = s;
  h->bank[bk].serial = ++h->stage_serial;
  PB = h->P;
  const bb_handle::Bank& B = h->bank[bk];
  PB.arena = B.arena; PB.st = B.st; PB.gkey = B.gkey; PB.gcoef = B.gcoef; PB.glen = B.glen; PB.gcount = B.gcount;
  PB.grlm = B.grlm; PB.gridx = B.gridx; PB.gflag = B.gflag;
  return bk;
}

// queries per pop of bb_reduce's workers: about four pops per worker, at most 32 queries each
#define BB_REDUCE_POPS 4
#define BB_REDUCE_CHUNK_MAX 32

int bb_reduce(bb_handle* h, int nlists, const int64_t* list_offsets_dev, const int64_t* poly_offsets_dev,
              const int32_t* exps_dev, const int32_t* coefs_dev, int nqueries, const int64_t* q_offsets_dev,
              const int32_t* q_exps_dev, const int32_t* q_coefs_dev, const int32_t* which_dev, int sorted, int32_t* steps_dev,
              int32_t* rlen_dev, int32_t* status_dev, const bb_poly_sink* rem, void* stream) {
  if (!h) return -1;
  if (nlists < 0 || nqueries < 0) return fail(h, "bb_reduce: negative count");
  if (!list_offsets_dev || !poly_offsets_dev || !exps_dev || !coefs_dev || !q_offsets_dev || !q_exps_dev || !q_coefs_dev ||
      !which_dev || !steps_dev || !rlen_dev || !status_dev)
    return fail(h, "bb_reduce: a required pointer is NULL");
  int rc = check_sink(h, rem, "rem", "bb_reduce");
  if (rc < 0) return rc;
  ENTER(h);
  if (nqueries == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  BBParams PB;
  const int bk = take_bank(h, s, PB);
  if (bk < 0) return bk;
  BBReduceArgs A;
  memset(&A, 0, sizeof A);
  A.nlists = nlists; A.nq = nqueries; A.sorted = sorted ? 1 : 0;
  A.chunk = (int)std::min<long long>(BB_REDUCE_CHUNK_MAX,
                                     std::max<long long>(1, nqueries / ((long long)BB_REDUCE_POPS * h->run_wave[0])));
  A.list_off = list_offsets_dev; A.poly_off = poly_offsets_dev; A.exps = exps_dev; A.coefs = coefs_dev;
  A.q_off = q_offsets_dev; A.q_exps = q_exps_dev; A.q_coefs = q_coefs_dev; A.which = which_dev;
  A.steps = steps_dev; A.rlen = rlen_dev; A.status = status_dev;
  if (rem) {
    A.sink = *rem;
    CK(cudaMemsetAsync(rem->where_dev, 0xff, sizeof(int64_t) * 2 * (size_t)nqueries, s));
  }
  A.queue = h->bank[bk].queue;
  CK(cudaMemsetAsync(A.queue, 0, sizeof(int), s));
  // workers: one per pop at most, no more than the bank's slots and the general runner's resident wave (same launch bounds)
  const int pops = (nqueries + A.chunk - 1) / A.chunk;
  const int workers = std::min(std::min(pops, h->P.num_envs), h->run_wave[0]);
  CK(h->K->reduce(PB, A, workers, s));
  CK(cudaEventRecord(h->bank[bk].done, s));
  return 0;
}

static int run_batches(bb_handle* h, int strategy, const BBPolicy* W, unsigned long long counter0, int episodes, int seed_base,
                       const int32_t* seeds_dev, int sel_seed_base, int max_steps, double gamma, int compute_gb,
                       bb_episode_stats* stats_dev, int32_t* trace_dev, int trace_episodes, int trace_cap, void* stream,
                       const bb_poly_sink* gb, const bb_poly_sink* basis);

int bb_run(bb_handle* h, int strategy, int episodes, int seed_base, const int32_t* seeds_dev, int sel_seed_base,
           int max_steps, double gamma, int compute_gb, bb_episode_stats* stats_dev, int32_t* trace_dev,
           int trace_episodes, int trace_cap, void* stream) {
  return bb_run_export(h, strategy, episodes, seed_base, seeds_dev, sel_seed_base, max_steps, gamma, compute_gb, stats_dev,
                       trace_dev, trace_episodes, trace_cap, stream, nullptr, nullptr);
}

int bb_run_export(bb_handle* h, int strategy, int episodes, int seed_base, const int32_t* seeds_dev, int sel_seed_base,
                  int max_steps, double gamma, int compute_gb, bb_episode_stats* stats_dev, int32_t* trace_dev,
                  int trace_episodes, int trace_cap, void* stream, const bb_poly_sink* gb, const bb_poly_sink* basis) {
  if (!h) return -1;
  if ((unsigned)strategy > 8u || episodes < 0 || !stats_dev) return fail(h, "bb_run: bad argument");
  if (gb && !compute_gb) return fail(h, "bb_run_export: a gb sink needs compute_gb != 0");
  int rc = check_sink(h, gb, "gb");
  if (rc == 0) rc = check_sink(h, basis, "basis");
  if (rc < 0) return rc;
  return run_batches(h, strategy, nullptr, 0, episodes, seed_base, seeds_dev, sel_seed_base, max_steps, gamma, compute_gb,
                     stats_dev, trace_dev, trace_episodes, trace_cap, stream, gb, basis);
}

// The body of bb_run_export and bb_run_policy (arguments already checked): batching, matching bb_prepare batches, the bank,
// staging and the sinks.  W == NULL: built-in selection `strategy` by the runner the handle's modes pick; otherwise the
// policy runner (k_run_policy) with weights W and step-0 counter counter0.
static int run_batches(bb_handle* h, int strategy, const BBPolicy* W, unsigned long long counter0, int episodes, int seed_base,
                       const int32_t* seeds_dev, int sel_seed_base, int max_steps, double gamma, int compute_gb,
                       bb_episode_stats* stats_dev, int32_t* trace_dev, int trace_episodes, int trace_cap, void* stream,
                       const bb_poly_sink* gb, const bb_poly_sink* basis) {
  ENTER(h);
  cudaStream_t s = (cudaStream_t)stream;
  if (episodes == 0) return 0;
  int rc = check_staged(h, W ? "bb_run_policy" : "bb_run");
  if (rc < 0) return rc;
  // the policy runner's resident wave for this hidden width (cached: it depends only on the handle's cols and on hidden)
  int policy_wave = 0;
  if (W) {
    int& w = h->policy_wave[W->hidden == 32 ? 0 : (W->hidden == 64 ? 1 : (W->hidden == 128 ? 2 : 3))];
    if (w == 0) {
      const int per_sm = h->K->run_policy_warps_per_sm(h->P, W->hidden);
      if (per_sm <= 0) return fail(h, "bb_run_policy: the policy runner does not fit this device");
      w = per_sm * h->sm_count;
    }
    policy_wave = w;
  }
  // long polynomials (general capacities): reduce() by streams with one CTA per environment (bb_wide.cuh: the shortest
  // chain of additions).  Modes 4 / 5 / 6 are kept for compatibility and run as 1 / 2 / 3.  The policy runner always steps
  // with the materialising reduction: its episodes are dominated by the head.
  const int mode = h->wide_mode >= 4 && h->wide_mode <= 6 ? h->wide_mode - 3 : h->wide_mode;
  const bool streams = !W && mode != 0 && (mode >= 1 || h->P.max_poly_terms >= 256);
  const int stream_kmax = mode == 2 ? 6 : (mode == 3 ? 48 : BBS_KMAX);
  const int stream_regs = mode == 7 ? 8 : stream_kmax;
  const int ctl_reducers = mode == 8 ? 32 : 256;
  int wide_ctas = 0;
  if (streams) {
    wide_ctas = h->K->wide_ctas_per_sm() * h->sm_count;
    if (wide_ctas <= 0) return fail(h, "bb_run: the CTA-per-environment stream runner does not fit this device");
  }
  const int nbatch = (episodes + BB_RUN_BATCH - 1) / BB_RUN_BATCH;
  BBParams PB;
  const int bk = take_bank(h, s, PB);
  if (bk < 0) return bk;
  // Batch 0: already prepared by a matching bb_prepare, or prepared here on the caller's stream.  Batches 1.. of the
  // same call are prepared on the handle's side stream while the runner works through their predecessor.
  int which = -1;
  {
    const int count0 = std::min(BB_RUN_BATCH, episodes);
    for (int b = 0; b < BB_STAGE_SETS; b++) {   // the oldest waiting batch that is this call's
      const bb_handle::Stage& T = h->stage[b];
      const bool m = T.episodes == count0 && nbatch == 1 && T.seed_base == seed_base && T.seeds == seeds_dev;
      if (m && (which < 0 || T.serial < h->stage[which].serial)) which = b;
    }
    const bool ready = which >= 0;
    if (!ready) which = stage_take(h);
    bb_handle::Stage& T = h->stage[which];
    if (h->timing) CK(cudaEventRecord(h->ev_t[0], s));
    if (ready) CK(cudaStreamWaitEvent(s, T.prepared, 0));
    else {
      rc = enqueue_prepare(h, which, 0, count0, seed_base, seeds_dev, s);
      if (rc < 0) return rc;
    }
    T.episodes = 0;
    if (h->timing) CK(cudaEventRecord(h->ev_t[1], s));
  }
  if (nbatch > 1) CK(cudaEventRecord(h->ev_entry, s));   // seeds_dev and the ideals are valid on the side stream from here on
  // where = (-1, -1) for every episode; the runners overwrite it for the episodes they store
  for (const bb_poly_sink* k : {gb, basis})
    if (k) CK(cudaMemsetAsync(k->where_dev, 0xff, sizeof(int64_t) * 2 * (size_t)episodes, s));
  for (int bi = 0; bi < nbatch; bi++) {
    const int base = bi * BB_RUN_BATCH, count = std::min(BB_RUN_BATCH, episodes - base);
    int next = -1;
    if (bi + 1 < nbatch) {   // the next batch into another set, concurrently with this batch's runner
      const int nbase = base + BB_RUN_BATCH;
      if (bi == 0) CK(cudaStreamWaitEvent(h->side, h->ev_entry, 0));
      next = stage_take(h);
      rc = enqueue_prepare(h, next, nbase, std::min(BB_RUN_BATCH, episodes - nbase), seed_base, seeds_dev, h->side);
      if (rc < 0) return rc;
    }
    BBParams S;
    rc = stage_params(h, which, h->stage[which].cap, S);
    if (rc < 0) return rc;
    BBRunArgs A;
    prepare_args(h, which, base, count, seed_base, seeds_dev, A);
    A.strategy = strategy; A.sel_seed_base = sel_seed_base; A.sel_seed_stride = h->sel_seed_stride;
    A.max_steps = max_steps; A.gamma = gamma; A.compute_gb = compute_gb; A.out = stats_dev;
    if (gb) A.gb_sink = *gb;
    if (basis) A.basis_sink = *basis;
    A.trace = trace_dev; A.trace_eps = trace_dev ? trace_episodes : 0; A.trace_cap = trace_cap;
    A.stream_kmax = stream_kmax; A.stream_regs = stream_regs; A.ctl_reducers = ctl_reducers;
    // every generator a binomial distribution draws has two terms, so every polynomial of the run has at most two
    // (DESIGN.md §3).  Staged ideals keep the general runner: nothing records the length of their polynomials.
    A.two_term = !W && h->two_term && h->P.dist.enabled && h->P.dist.kind == 0;
    if (bi > 0) CK(cudaStreamWaitEvent(s, h->stage[which].prepared, 0));
    const int workers = std::min(h->P.num_envs, count);
    if (W) CK(h->K->run_policy(PB, S, A, *W, counter0, std::min(workers, policy_wave), s));
    else if (streams) CK(h->K->run_wide(PB, S, A, std::min(workers, wide_ctas), s));
    else CK(h->K->run(PB, S, A, std::min(workers, h->run_wave[A.two_term]), s));
    CK(cudaEventRecord(h->stage[which].consumed, s));
    CK(cudaEventRecord(h->bank[bk].done, s));
    if (h->timing && bi == 0) CK(cudaEventRecord(h->ev_t[2], s));
    which = next;
  }
  return 0;
}

int bb_set_timing(bb_handle* h, int on) {
  if (!h) return -1;
  h->timing = on ? 1 : 0;
  return 0;
}

int bb_last_run_ms(bb_handle* h, float* prepare_ms, float* run_ms) {
  if (!h) return -1;
  if (!h->timing) return fail(h, "bb_last_run_ms: timing is off (bb_set_timing)");
  ENTER(h);
  CK(cudaEventSynchronize(h->ev_t[2]));
  float a = 0.f, b = 0.f;
  CK(cudaEventElapsedTime(&a, h->ev_t[0], h->ev_t[1]));
  CK(cudaEventElapsedTime(&b, h->ev_t[1], h->ev_t[2]));
  if (prepare_ms) *prepare_ms = a;
  if (run_ms) *run_ms = b;
  return 0;
}

int bb_set_episode_offset(bb_handle* h, int offset) {
  if (!h) return -1;
  if (offset < 0) return fail(h, "bb_set_episode_offset: negative offset");
  h->episode_offset = offset;
  return 0;
}

// Fork arena: `workers` full-size slots (same layout as the handle's own), allocated on first use and kept.
static int fork_params(bb_handle* h, int workers, BBParams& F) {
  const BBParams& P = h->P;
  F = P;
  if (workers > h->fork_cap) {
    for (void* p : h->fork_allocs) cudaFree(p);
    h->fork_allocs.clear();
    h->fork_cap = 0;
    auto alloc = [&](void** out, size_t bytes) {
      cudaError_t e = cudaMalloc(out, bytes + 16);
      if (e == cudaSuccess) { h->fork_allocs.push_back(*out); e = cudaMemset(*out, 0, bytes + 16); }
      return e;
    };
    CK(alloc((void**)&h->fork_arena, (size_t)workers * P.slot_stride));
    CK(alloc((void**)&h->fork_st, (size_t)workers * sizeof(BBEnvState)));
    h->fork_cap = workers;
  }
  F.arena = h->fork_arena; F.st = h->fork_st; F.num_envs = workers;
  return 0;
}

int bb_value(bb_handle* h, int strategy, double gamma, int rollouts, int sel_seed_base, int max_steps,
             double* value_dev, void* stream) {
  if (!h) return -1;
  if (!value_dev) return fail(h, "bb_value: null output");
  if (strategy == BB_VALUE_SAMPLE) rollouts = rollouts > 0 ? rollouts : 101;  // 1 Degree + 100 Random (buchberger.cpp:333-341)
  else if ((unsigned)strategy > 8u) return fail(h, "bb_value: bad strategy");
  else if (strategy != BB_SELECT_RANDOM || rollouts < 1) rollouts = 1;
  ENTER(h);
  cudaStream_t s = (cudaStream_t)stream;
  const int N = h->P.num_envs;
  const long long ntasks = (long long)N * rollouts;
  if (ntasks > 0x7fffffffLL) return fail(h, "bb_value: too many rollouts");
  // workers: one resident wave at most, and at most 8 GiB of fork arena
  int workers = h->run_wave[0];   // k_value has the general k_run's launch bounds
  const long long by_mem = (long long)(((size_t)8 << 30) / h->P.slot_stride);
  workers = (int)std::max(1LL, std::min((long long)workers, std::min(ntasks, by_mem)));
  BBParams F;
  if (workers > h->fork_cap) CK(cudaStreamSynchronize(s));
  int rc = fork_params(h, std::max(workers, h->fork_cap), F);
  if (rc < 0) return rc;
  F.num_envs = workers;
  BBValueArgs A;
  A.strategy = strategy; A.rollouts = rollouts; A.sel_seed_base = sel_seed_base; A.max_steps = max_steps;
  A.gamma = gamma; A.value = value_dev; A.queue = h->d_queue; A.ntasks = (int)ntasks;
  CK(cudaMemsetAsync(h->d_queue, 0, sizeof(int), s));
  k_fill_double<<<(N + BB_THREADS - 1) / BB_THREADS, BB_THREADS, 0, s>>>(value_dev, N, -__builtin_inf());
  CK(cudaGetLastError());
  CK(h->K->value(h->P, F, A, workers, s));
  return 0;
}

// BuchbergerEnv copy constructor (buchberger.cpp:279-283; wrapped.pyx:35-38 copy()): the whole environment --
// basis, pair set, reducer list, staged ideal, both random streams and the episode record.
int bb_copy_env(bb_handle* dst, int dst_env, bb_handle* src, int src_env, void* stream) {
  bb_handle* h = dst;
  if (!dst || !src) return -1;
  if (dst_env < 0 || dst_env >= dst->P.num_envs || src_env < 0 || src_env >= src->P.num_envs)
    return fail(h, "bb_copy_env: environment index out of range");
  const bb_config &a = dst->cfg, &b = src->cfg;
  if (a.device != b.device || a.nvars != b.nvars || a.prime != b.prime || a.max_basis != b.max_basis ||
      a.max_pairs != b.max_pairs || a.max_terms != b.max_terms || a.max_poly_terms != b.max_poly_terms ||
      a.max_gens != b.max_gens || a.max_gen_terms != b.max_gen_terms)
    return fail(h, "bb_copy_env: handles differ in device, field, variables or capacities");
  if (dst == src && dst_env == src_env) return 0;
  CK(cudaSetDevice(a.device));
  if (dst->serving) { int rc = serve_stop(dst); if (rc < 0) return rc; }
  if (src->serving && serve_stop(src) < 0) return fail(h, "bb_copy_env: " + src->err);
  cudaStream_t s = (cudaStream_t)stream;
  const BBParams &D = dst->P, &S = src->P;
  CK(cudaMemcpyAsync(D.arena + (size_t)dst_env * D.slot_stride, S.arena + (size_t)src_env * S.slot_stride, S.slot_stride,
                     cudaMemcpyDeviceToDevice, s));
  CK(cudaMemcpyAsync(D.st + dst_env, S.st + src_env, sizeof(BBEnvState), cudaMemcpyDeviceToDevice, s));
  CK(cudaMemcpyAsync(D.in_key + (size_t)dst_env * D.max_gen_terms, S.in_key + (size_t)src_env * S.max_gen_terms,
                     sizeof(uint64_t) * S.max_gen_terms, cudaMemcpyDeviceToDevice, s));
  CK(cudaMemcpyAsync(D.in_coef + (size_t)dst_env * D.max_gen_terms, S.in_coef + (size_t)src_env * S.max_gen_terms,
                     sizeof(uint32_t) * S.max_gen_terms, cudaMemcpyDeviceToDevice, s));
  CK(cudaMemcpyAsync(D.in_off + (size_t)dst_env * (D.max_gens + 1), S.in_off + (size_t)src_env * (S.max_gens + 1),
                     sizeof(int) * (S.max_gens + 1), cudaMemcpyDeviceToDevice, s));
  CK(cudaMemcpyAsync(D.in_np + dst_env, S.in_np + src_env, sizeof(int), cudaMemcpyDeviceToDevice, s));
  if (dst->pre_ready) {   // the destination's prepared episodes belonged to its old stream
    k_pre_flush<<<(D.num_envs + BB_THREADS - 1) / BB_THREADS, BB_THREADS, 0, s>>>(D, dst_env);
    CK(cudaGetLastError());
  }
  return 0;
}

int bb_discount(bb_handle* h, int N, int T, const double* x_dev, const uint8_t* done_dev, double gam, double* out_dev,
                void* stream) {
  if (!h) return -1;
  if (N < 0 || T < 0 || !x_dev || !done_dev || !out_dev) return fail(h, "bb_discount: bad argument");
  if (N == 0 || T == 0) return 0;
  ENTER(h);
  k_discount<<<(N + BB_THREADS - 1) / BB_THREADS, BB_THREADS, 0, (cudaStream_t)stream>>>(N, T, x_dev, done_dev, gam, out_dev);
  CK(cudaGetLastError());
  return 0;
}

int bb_set_prefetch(bb_handle* h, int depth) {
  if (!h) return -1;
  if (depth < 0 || depth > 64) return fail(h, "bb_set_prefetch: depth must be in 0..64");
  ENTER(h);
  if (h->pre_ready) { CK(cudaDeviceSynchronize()); pre_drop(h); }
  h->pre_depth = depth;
  return 0;
}

int bb_set_serve(bb_handle* h, int on) {
  if (!h) return -1;
  ENTER(h);
  h->serve_on = on ? 1 : 0;
  return 0;
}

int bb_set_compaction(bb_handle* h, int on) {
  if (!h) return -1;
  h->compaction = on ? 1 : 0;
  return 0;
}

int bb_compact(bb_handle* h, int32_t* active_dev, void* stream) {
  if (!h) return -1;
  ENTER(h);
  cudaStream_t s = (cudaStream_t)stream;
  k_compact<<<1, 1024, 0, s>>>(h->P, active_dev ? active_dev : h->d_active);
  CK(cudaGetLastError());
  return 0;
}

int bb_status_summary(bb_handle* h, int32_t* counts_host, void* stream) {
  if (!h || !counts_host) return -1;
  ENTER(h);
  cudaStream_t s = (cudaStream_t)stream;
  int* hist = h->d_active;   // the list is rebuilt by every call that uses it
  CK(cudaMemsetAsync(hist, 0, sizeof(int) * BB_STATUS_COUNT, s));
  k_status_hist<<<(h->P.num_envs + BB_THREADS - 1) / BB_THREADS, BB_THREADS, 0, s>>>(h->P, hist);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(counts_host, hist, sizeof(int) * BB_STATUS_COUNT, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  return 0;
}

int bb_set_max_episode_length(bb_handle* h, int max_steps) {
  if (!h) return -1;
  if (max_steps < 0) return fail(h, "bb_set_max_episode_length: negative length");
  ENTER(h);
  h->P.max_episode_length = max_steps;
  return 0;
}

int bb_set_obs_nvars(bb_handle* h, int n_obs) {
  if (!h) return -1;
  if (n_obs < 1 || n_obs > h->cfg.nvars) return fail(h, "bb_set_obs_nvars: must be in 1..nvars");
  ENTER(h);
  h->P.obs_nv = n_obs;
  h->P.cols = 2 * n_obs * h->P.k;
  return 0;
}

int bb_set_wide(bb_handle* h, int mode) {
  if (!h) return -1;
  if (mode < -1 || mode > 8) return fail(h, "bb_set_wide: mode must be -1 (auto), 0 (off), 1 (on), 2 or 3 (on, 6 / 48 stream slots), 4, 5 or 6 (as 1, 2 or 3), 7 (as 1, 8 register slots + the shared-memory table), 8 (as 1, 32 reducers in the control warp's registers)");
  h->wide_mode = mode;
  return 0;
}

int bb_set_prepare_mode(bb_handle* h, int by_warp) {
  if (!h) return -1;
  h->prepare_by_warp = by_warp ? 1 : 0;
  return 0;
}

int bb_set_two_term(bb_handle* h, int on) {
  if (!h) return -1;
  h->two_term = on ? 1 : 0;
  return 0;
}

int bb_set_selection_seed_stride(bb_handle* h, int stride) {
  if (!h) return -1;
  h->sel_seed_stride = stride;
  return 0;
}

int bb_set_auto_reset(bb_handle* h, int on) {
  if (!h) return -1;
  ENTER(h);
  h->P.auto_reset = on ? 1 : 0;
  return 0;
}

static int check_policy(bb_handle* h, int hidden, const float* W1, const float* b1, const float* w2, const float* b2) {
  if (!W1 || !b1 || !w2 || !b2) return fail(h, "policy: null weight pointer");
  if (hidden != 32 && hidden != 64 && hidden != 128 && hidden != 256) return fail(h, "policy: hidden must be 32, 64, 128 or 256");
  if (h->P.cols > BB_POLICY_MAX_COLS) return fail(h, "policy: more than 64 state columns");
  if (h->P.obs_nv != h->P.nvars) return fail(h, "policy: not available under bb_set_obs_nvars (comparison mode of the state matrix)");
  return 0;
}

int bb_policy_pmlp(bb_handle* h, int hidden, const float* W1_dev, const float* b1_dev, const float* w2_dev,
                   const float* b2_dev, uint64_t seed, uint64_t counter, int greedy, int32_t* actions_dev,
                   float* logprob_dev, float* logprobs_all_dev, int pmax, void* stream) {
  if (!h) return -1;
  int rc = check_policy(h, hidden, W1_dev, b1_dev, w2_dev, b2_dev);
  if (rc < 0) return rc;
  if (!actions_dev || (logprobs_all_dev && pmax < 1)) return fail(h, "bb_policy_pmlp: bad argument");
  ENTER(h);
  BBPolicy W;
  W.hidden = hidden; W.W1 = W1_dev; W.b1 = b1_dev; W.w2 = w2_dev; W.b2 = b2_dev; W.seed = seed; W.greedy = greedy ? 1 : 0;
  CK(h->K->policy(h->P, W, counter, actions_dev, logprob_dev, logprobs_all_dev, pmax, h->P.num_envs, (cudaStream_t)stream));
  return 0;
}

int bb_rollout(bb_handle* h, int hidden, const float* W1_dev, const float* b1_dev, const float* w2_dev, const float* b2_dev,
               uint64_t seed, uint64_t counter0, int greedy, int T, int32_t* actions_dev, float* logprob_dev,
               float* reward_dev, uint8_t* done_dev, int32_t* lengths_dev, int32_t* obs_dev, int pmax, void* stream) {
  return bb_rollout_value(h, hidden, W1_dev, b1_dev, w2_dev, b2_dev, seed, counter0, greedy, T, actions_dev, logprob_dev,
                          reward_dev, done_dev, lengths_dev, obs_dev, pmax, BB_SELECT_DEGREE, 0.99, 1, 0, 0, nullptr, stream);
}

int bb_rollout_value(bb_handle* h, int hidden, const float* W1_dev, const float* b1_dev, const float* w2_dev,
                     const float* b2_dev, uint64_t seed, uint64_t counter0, int greedy, int T, int32_t* actions_dev,
                     float* logprob_dev, float* reward_dev, uint8_t* done_dev, int32_t* lengths_dev, int32_t* obs_dev, int pmax,
                     int value_strategy, double value_gamma, int value_rollouts, int value_sel_seed, int value_max_steps,
                     double* value_dev, void* stream) {
  return bb_rollout_rows(h, hidden, W1_dev, b1_dev, w2_dev, b2_dev, seed, counter0, greedy, T, actions_dev, logprob_dev,
                         reward_dev, done_dev, lengths_dev, obs_dev, pmax, value_strategy, value_gamma, value_rollouts,
                         value_sel_seed, value_max_steps, value_dev, nullptr, 0, stream);
}

int bb_rollout_rows(bb_handle* h, int hidden, const float* W1_dev, const float* b1_dev, const float* w2_dev,
                    const float* b2_dev, uint64_t seed, uint64_t counter0, int greedy, int T, int32_t* actions_dev,
                    float* logprob_dev, float* reward_dev, uint8_t* done_dev, int32_t* lengths_dev, int32_t* obs_dev, int pmax,
                    int value_strategy, double value_gamma, int value_rollouts, int value_sel_seed, int value_max_steps,
                    double* value_dev, int32_t* rows_dev, int64_t rows_per_env, void* stream) {
  if (!h) return -1;
  int rc = check_policy(h, hidden, W1_dev, b1_dev, w2_dev, b2_dev);
  if (rc < 0) return rc;
  if (T < 1 || (obs_dev && pmax < 1)) return fail(h, "bb_rollout: bad argument");
  // every environment can store the state it starts the call from
  if (rows_dev && rows_per_env < h->P.max_pairs) return fail(h, "bb_rollout_rows: rows_per_env is below max_pairs");
  // bb_value's rules
  if (value_strategy == BB_VALUE_SAMPLE) value_rollouts = value_rollouts > 0 ? value_rollouts : 101;
  else if ((unsigned)value_strategy > 8u) return fail(h, "bb_rollout_value: bad value strategy");
  else if (value_strategy != BB_SELECT_RANDOM || value_rollouts < 1) value_rollouts = 1;
  ENTER(h);
  cudaStream_t s = (cudaStream_t)stream;
  BBRolloutArgs A;
  A.W.hidden = hidden; A.W.W1 = W1_dev; A.W.b1 = b1_dev; A.W.w2 = w2_dev; A.W.b2 = b2_dev; A.W.seed = seed;
  A.W.greedy = greedy ? 1 : 0;
  A.T = T; A.counter0 = counter0; A.actions = actions_dev; A.logp = logprob_dev; A.reward = reward_dev; A.done = done_dev;
  A.lengths = lengths_dev; A.obs = obs_dev; A.pmax = pmax; A.rows = rows_dev; A.rows_per_env = rows_dev ? rows_per_env : 0;
  A.rows_budget = (int)std::min<int64_t>(A.rows_per_env, INT_MAX);
  BBParams F;
  BBValueArgs V;
  if (value_dev) {   // one fork slot per environment: environment e's value rollouts run in slot e
    const int N = h->P.num_envs;
    if ((long long)N > (long long)(((size_t)8 << 30) / h->P.slot_stride))
      return fail(h, "bb_rollout_value: the fork arena (one slot per environment) would exceed 8 GiB");
    if (N > h->fork_cap) CK(cudaStreamSynchronize(s));
    rc = fork_params(h, std::max(N, h->fork_cap), F);
    if (rc < 0) return rc;
    F.num_envs = N;
    V.strategy = value_strategy; V.rollouts = value_rollouts; V.sel_seed_base = value_sel_seed; V.max_steps = value_max_steps;
    V.gamma = value_gamma; V.value = value_dev; V.queue = nullptr; V.ntasks = 0;
  }
  if (h->P.auto_reset) { rc = pre_refill(h, s, true); if (rc < 0) return rc; }
  CK(h->K->rollout(h->P, A, value_dev ? &F : nullptr, value_dev ? &V : nullptr, h->P.num_envs, s));
  return 0;
}

int bb_run_policy(bb_handle* h, int hidden, const float* W1_dev, const float* b1_dev, const float* w2_dev,
                  const float* b2_dev, uint64_t seed, uint64_t counter0, int greedy,
                  int episodes, int seed_base, const int32_t* seeds_dev, int max_steps, double gamma, int compute_gb,
                  bb_episode_stats* stats_dev, int32_t* trace_dev, int trace_episodes, int trace_cap, void* stream,
                  const bb_poly_sink* gb, const bb_poly_sink* basis) {
  if (!h) return -1;
  int rc = check_policy(h, hidden, W1_dev, b1_dev, w2_dev, b2_dev);
  if (rc < 0) return rc;
  if (episodes < 0 || !stats_dev) return fail(h, "bb_run_policy: bad argument");
  if (gb && !compute_gb) return fail(h, "bb_run_policy: a gb sink needs compute_gb != 0");
  rc = check_sink(h, gb, "gb", "bb_run_policy");
  if (rc == 0) rc = check_sink(h, basis, "basis", "bb_run_policy");
  if (rc < 0) return rc;
  BBPolicy W;
  W.hidden = hidden; W.W1 = W1_dev; W.b1 = b1_dev; W.w2 = w2_dev; W.b2 = b2_dev; W.seed = seed; W.greedy = greedy ? 1 : 0;
  return run_batches(h, 0, &W, counter0, episodes, seed_base, seeds_dev, 0, max_steps, gamma, compute_gb, stats_dev, trace_dev,
                     trace_episodes, trace_cap, stream, gb, basis);
}

static int unpack_polys(bb_handle* h, const std::vector<uint64_t>& keys, const std::vector<uint32_t>& cf,
                        const std::vector<int>& plen, int32_t* lens, int cap_polys, int32_t* exps, int32_t* coefs,
                        int cap_terms, int* nterms_out) {
  const BBLayout& L = h->L;
  int np = (int)plen.size(), nt = 0;
  for (int q = 0; q < np; q++) nt += plen[q];
  if (nterms_out) *nterms_out = nt;
  if (np > cap_polys || nt > cap_terms) return fail(h, "output buffers too small", -4);
  for (int q = 0; q < np; q++) lens[q] = plen[q];
  for (int t = 0; t < nt; t++) {
    coefs[t] = (int32_t)cf[t];
    for (int v = 0; v < L.n; v++) exps[(size_t)t * L.n + v] = (int32_t)bb_exp(L, keys[t], v);
  }
  return np;
}

int bb_download_basis(bb_handle* h, int env, int32_t* lens, int cap_polys, int32_t* exps, int32_t* coefs,
                      int cap_terms, int* nterms_out) {
  if (!h) return -1;
  BBParams& P = h->P;
  if (env < 0 || env >= P.num_envs) return fail(h, "bb_download_basis: environment index out of range");
  ENTER(h);
  CK(cudaDeviceSynchronize());
  BBEnvState S;
  CK(cudaMemcpy(&S, P.st + env, sizeof S, cudaMemcpyDeviceToHost));
  std::vector<GHeadMem> meta((size_t)std::max(S.nG, 1));
  std::vector<uint64_t> keys((size_t)std::max(S.nT, 1));
  std::vector<uint32_t> cf((size_t)std::max(S.nT, 1));
  const unsigned char* base = P.arena + (size_t)env * P.slot_stride;
  if (S.nG) CK(cudaMemcpy(meta.data(), base + P.o_ghead, sizeof(GHeadMem) * S.nG, cudaMemcpyDeviceToHost));
  if (S.nT) {
    CK(cudaMemcpy(keys.data(), base + P.o_tkey, sizeof(uint64_t) * S.nT, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(cf.data(), base + P.o_tcoef, sizeof(uint32_t) * S.nT, cudaMemcpyDeviceToHost));
  }
  // polynomials are stored back to back in insertion order
  std::vector<int> plen;
  for (int q = 0; q < S.nG; q++) plen.push_back((int)meta[q].len);
  return unpack_polys(h, keys, cf, plen, lens, cap_polys, exps, coefs, cap_terms, nterms_out);
}

int bb_final_gb(bb_handle* h, int env, int32_t* lens, int cap_polys, int32_t* exps, int32_t* coefs, int cap_terms,
                int* nterms_out) {
  if (!h) return -1;
  BBParams& P = h->P;
  if (env < 0 || env >= P.num_envs) return fail(h, "bb_final_gb: environment index out of range");
  ENTER(h);
  CK(h->K->final_gb(P, env, h->d_ok, (cudaStream_t)0));
  CK(cudaDeviceSynchronize());
  int ok = 0, cnt[2] = {0, 0};
  CK(cudaMemcpy(&ok, h->d_ok, sizeof(int), cudaMemcpyDeviceToHost));
  if (!ok) return fail(h, "bb_final_gb: arena overflow while interreducing", -5);
  CK(cudaMemcpy(cnt, P.gcount + 2 * (size_t)env, sizeof cnt, cudaMemcpyDeviceToHost));
  std::vector<int> plen((size_t)cnt[0]);
  std::vector<uint64_t> keys((size_t)std::max(cnt[1], 1));
  std::vector<uint32_t> cf((size_t)std::max(cnt[1], 1));
  if (cnt[0]) CK(cudaMemcpy(plen.data(), P.glen + (size_t)env * P.max_basis, sizeof(int) * cnt[0], cudaMemcpyDeviceToHost));
  if (cnt[1]) {
    CK(cudaMemcpy(keys.data(), P.gkey + (size_t)env * P.max_terms, sizeof(uint64_t) * cnt[1], cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(cf.data(), P.gcoef + (size_t)env * P.max_terms, sizeof(uint32_t) * cnt[1], cudaMemcpyDeviceToHost));
  }
  return unpack_polys(h, keys, cf, plen, lens, cap_polys, exps, coefs, cap_terms, nterms_out);
}

int bb_counters_read(bb_handle* h, bb_counters* out, int reset) {
  if (!h || !out) return -1;
  ENTER(h);
  CK(cudaDeviceSynchronize());
  unsigned long long v[CT_COUNT];
  CK(cudaMemcpy(v, h->P.counters, sizeof v, cudaMemcpyDeviceToHost));
  out->env_steps = v[CT_STEPS]; out->additions = v[CT_ADDS]; out->terms_read = v[CT_TREAD];
  out->terms_written = v[CT_TWRITE]; out->lms_scanned = v[CT_LMS]; out->term_moves = v[CT_MOVES];
  out->update_basis = v[CT_UPB]; out->update_pairs = v[CT_UPP]; out->obs_rows = v[CT_OBS];
  out->nonzero_reductions = v[CT_NONZERO]; out->zero_reductions = v[CT_ZERO]; out->episodes = v[CT_EPISODES];
  if (reset) CK(cudaMemset(h->P.counters, 0, sizeof v));
  return 0;
}

}  // extern "C"
