// bb_kernels.cuh -- the kernels of libbbenv.so, templated on the number of variables NV (compile-time monomial
// layout), and the per-NV launch table the host API (bbenv.cu) dispatches through.  sm_100a only.
//
// Kernels (one warp per environment slot, BB_WARPS warps per CTA):
//   k_reset    BuchbergerEnv::reset          buchberger.cpp:299-315  (+ on-device ideal generator, ideals.cpp:168-201)
//   k_step     LeadMonomialsEnv::step(int)   buchberger.cpp:398-408 -> :318-329 (spoly, reduce, update, insert)
//   k_select   First/Degree/Normal           buchberger.cpp:165-186
//   k_observe  state matrix                  buchberger.cpp:354-370, 402-406
//   k_run      persistent: episodes pulled from a queue and run to completion with on-device selection
//              (the loop of buchberger(), buchberger.cpp:243-263); finished slots refill at once.
//   k_run_policy the same runner with the pairs policy head (bb_policy.cuh) choosing the pairs (bb_run_policy)
//   k_run_wide the same runner with one CTA per environment slot and reduce() by streams (bb_wide.cuh: long polynomials)
//   k_final_gb interreduce(minimalize(G))    buchberger.cpp:102-122
//   k_reduce   reduce(g, F)                  buchberger.cpp:24-49 on caller-supplied divisor lists and dividends (bb_reduce)
#pragma once
#include <type_traits>

#include "bb_device.cuh"
#include "bb_policy.cuh"
#if defined(BBW_CLOCK) || defined(BBW_INSTR)
#include <cstdio>
#endif
#include "bb_wide.cuh"

#ifndef BB_WARPS
#define BB_WARPS 8
#endif
#define BB_THREADS (BB_WARPS * 32)
#ifndef BB_MIN_BLOCKS
#define BB_MIN_BLOCKS 3  // register cap 80 -> 24 resident warps per SM: the general k_run (A/B on B200, profiles/README.md v8: 2 -> 702, 3 -> 763, 4 -> 728, 5 -> 693, 6 -> 657 M env-steps/s) and the step kernels
#endif
// The two-term k_run (k_run<NV, EXPORT, true>) has launch bounds of its own: it spills far less than the general runner
// under a lower register cap, so it keeps more warps resident
// (profiles/README.md, "Two-term runner at 32 warps per SM": 8 x 4 against 8 x 3, 7 x 4, 6 x 5 and 4 x 8).
#ifndef BB_TWO_WARPS
#define BB_TWO_WARPS BB_WARPS
#endif
#ifndef BB_TWO_MIN_BLOCKS
#define BB_TWO_MIN_BLOCKS 4  // register cap 64 -> 32 resident warps per SM
#endif

#ifndef BB_ROLLOUT_MIN_BLOCKS
#define BB_ROLLOUT_MIN_BLOCKS 2  // 128 registers, no spills, 16 warps/SM: 140 M env-steps/s against 132 M at 3 and 123 M at 4 (profiles/README.md v10)
#endif

struct BBRunArgs {
  int strategy, episodes, seed_base;
  int sel_seed_base;  // Random selection: episode e draws choice() from minstd_rand0 seeded sel_seed_base + e * sel_seed_stride
  int sel_seed_stride;
  int ep_base;      // first episode of this batch: episode ids are ep_base .. ep_base + episodes - 1
  int ep_offset;    // global index of the call's episode 0 (bb_set_episode_offset): selection seeds and the staged ideal
                    // an episode replays follow the GLOBAL index, so a shard of a job behaves like its slice of the whole
  int nstaged;      // fixed ideals: number of staged ideals (global episode g replays ideal g mod nstaged)
  const int* seeds;
  int max_steps;
  double gamma;
  int compute_gb;
  bb_poly_sink gb_sink, basis_sink;   // bb_run_export (lens_dev == NULL: no sink); where_dev is indexed by ep_base + b
  bb_episode_stats* out;
  int32_t* trace;
  int trace_eps, trace_cap;
  int prepare_by_warp;  // 1: k_prepare (one warp per episode) even where k_prepare_lanes applies (tests compare the two)
  int stream_kmax;   // k_run_wide: stream slots a step's reduction may use (BBS_KMAX; 6 / 48 under bb_set_wide(2 / 3)), see bb_wide.cuh
  int stream_regs;   // k_run_wide: how many of them are register slots (BBW_SLOTS; 8 under bb_set_wide(7))
  int ctl_reducers;  // k_run_wide: reducers of G_ in the control warp's registers (256; 32 under bb_set_wide(8))
  int* queue;        // [0]: next queue position; [BB_LPT_HIST .. +BB_LPT_BUCKETS): histogram of the cost keys of the batch, then as many cursors
  int* order;        // [episodes] queue position -> episode of the batch, longest predicted first (k_order)
  uint8_t* cost_key; // [episodes] predicted-cost bucket of each episode of the batch (k_prepare)
  int two_term;      // k_run: every polynomial has at most two terms (binomial ideals): the two-term instantiation
};
#define BB_LPT_BUCKETS 256
#define BB_LPT_HIST 4

// Prefetch queues of the step API.  reset() inside a step kernel (auto-reset) is a cold detour of one warp through the ideal
// generator and s update() calls: 38 us, while the other warps of the launch wait for it at the kernel's end.  Instead every
// environment keeps a short queue of its NEXT episodes' initial states, prepared in bulk by k_prefill (one thread per
// environment, k_prepare_lanes' code) from the environment's own ideal stream, in stream order; a reset takes the head of the
// queue with a copy.  st.rng stays the stream position after the CURRENT episode's draw (= before the head of the queue), so
// dropping a queue (seed(), copy()) never changes what an environment draws next.  Lives in device memory; P.pre points at it.
#define BB_PREP_S 16   // most generators the thread-per-episode preparation handles
struct BBPre {
  BBParams S;        // staging-layout parameters of the queue slots: slot (e * depth + j)
  int depth;
  int* count;        // [num_envs] episodes waiting
  int* head;         // [num_envs] position of the first one
  unsigned* rng;     // [num_envs] stream state after the LAST prepared episode (where k_prefill goes on)
  int* calls;        // [1] step calls so far (ticked by k_step / k_step_obs): k_prefill, launched with every call, works every
                     // `period`-th one only -- the decision is taken on the device so that it survives CUDA-graph replay
};

struct BBEpisodeAcc {
  unsigned long long th;
  double ret, disc;
  uint32_t sel_rng, pad;
};

struct BBValueArgs {
  int strategy;       // BB_SELECT_* or BB_VALUE_SAMPLE
  int rollouts;       // rollouts per environment (max of their returns); SAMPLE: 1 Degree + (rollouts - 1) Random
  int sel_seed_base;  // Random rollout r is seeded sel_seed_base + r (SAMPLE: sel_seed_base + r - 1)
  int max_steps;
  double gamma;
  double* value;      // [num_envs], pre-filled with -inf
  int* queue;
  int ntasks;         // num_envs * rollouts
};

struct BBRolloutArgs {
  BBPolicy W;
  int T;                          // steps per environment
  unsigned long long counter0;    // step t draws its uniform from (seed + env, counter0 + t)
  // outputs, all [N, T] (environment-major: one trajectory is contiguous); any may be NULL
  int32_t* actions; float* logp; float* reward; uint8_t* done; int32_t* lengths;
  int32_t* obs; int pmax;         // optional [N, T, pmax, cols] state matrices BEFORE each step, padded with -1
};

// Mailbox of the single-environment server (k_serve), in mapped pinned host memory.  The host writes a command and bumps
// cmd_seq; the resident warp polls cmd_seq over PCIe, executes, writes the results (the state matrix behind the header) and
// publishes done_seq = cmd_seq.  alive: 1 while an instance of the kernel polls.
enum { BB_CMD_STEP = 1, BB_CMD_RESET = 2, BB_CMD_OBSERVE = 3, BB_CMD_STOP = 4 };
struct BBMailbox {
  // one 16-byte word, read by the device with ONE load (one PCIe round trip per poll, and the command comes with it)
  volatile unsigned cmd_seq;
  unsigned cmd;
  int arg;            // STEP: the action
  int rows;           // (rows of the state matrix to write, 0: none) << 1 | pad (rows beyond |P| are -1)
  unsigned pad0[12];
  volatile unsigned done_seq;   // second 64-byte line: written by the device
  volatile unsigned alive;
  int length;         // |P| after the command
  unsigned done;
  double reward;
  unsigned pad1[10];
  // int32 obs[pmax * cols] follows
};
static_assert(sizeof(BBMailbox) == 128, "mailbox header is two 64-byte lines");

// bb_reduce: caller-supplied divisor lists (PolyBatch layout: list -> polynomials -> terms, int64 offsets) and dividends.
// Queries come grouped by list; a worker warp pops `chunk` consecutive queries at a time and restages its slot only when
// the list changes.
struct BBReduceArgs {
  int nlists, nq, sorted, chunk;
  const int64_t* list_off; const int64_t* poly_off; const int32_t* exps; const int32_t* coefs;
  const int64_t* q_off; const int32_t* q_exps; const int32_t* q_coefs; const int32_t* which;
  int32_t* steps; int32_t* rlen; int32_t* status;
  bb_poly_sink sink;   // lens_dev == NULL: no sink
  int* queue;          // [1] next query, zeroed by the caller
};

struct BBKernelTable {
  int nvars, w, dw, dshift, eshift;
  cudaError_t (*reset)(const BBParams&, const uint8_t* mask, int nwarps, cudaStream_t);
  cudaError_t (*step)(const BBParams&, const int* actions, double* reward, uint8_t* done, const int* active, int nwarps,
                      cudaStream_t);
  cudaError_t (*step_obs)(const BBParams&, const int* actions, int action0, double* reward, uint8_t* done, int32_t* obs,
                          int32_t* lengths, int pmax, int pad, int do_step, const int* active, unsigned* ready, unsigned ticket,
                          int nwarps, cudaStream_t);
  cudaError_t (*serve)(const BBParams&, BBMailbox* mb, unsigned long long idle_ns, cudaStream_t);
  cudaError_t (*prefill)(const BBParams&, const BBParams& stage, int period, cudaStream_t);
  cudaError_t (*select)(const BBParams&, int strategy, int* actions, int nwarps, cudaStream_t);
  cudaError_t (*observe)(const BBParams&, int32_t* obs, int32_t* lengths, int pmax, int nwarps, cudaStream_t);
  cudaError_t (*final_gb)(const BBParams&, int slot, int* ok_out, cudaStream_t);
  cudaError_t (*prepare)(const BBParams& stage, const BBRunArgs&, cudaStream_t);  // k_prepare + k_order
  cudaError_t (*run)(const BBParams&, const BBParams& stage, const BBRunArgs&, int nwarps, cudaStream_t);
  // the same runner with reduce() by streams and one CTA per environment (bb_wide.cuh: long polynomials); nctas worker CTAs
  cudaError_t (*run_wide)(const BBParams&, const BBParams& stage, const BBRunArgs&, int nctas, cudaStream_t);
  int (*wide_ctas_per_sm)(void);
  cudaError_t (*value)(const BBParams&, const BBParams& fork, const BBValueArgs&, int nwarps, cudaStream_t);
  cudaError_t (*policy)(const BBParams&, const BBPolicy&, unsigned long long counter, int32_t* actions, float* logp,
                        float* logits, int pmax, int nwarps, cudaStream_t);
  cudaError_t (*rollout)(const BBParams&, const BBRolloutArgs&, int nwarps, cudaStream_t);
  int (*run_warps_per_sm)(int two);   // k_run: general (0) or two-term (1); -1 on error
  cudaError_t (*reduce)(const BBParams&, const BBReduceArgs&, int nwarps, cudaStream_t);
  // k_run with the policy head selecting (bb_run_policy), and its resident warps per SM for P.cols and W.hidden (-1 on error)
  cudaError_t (*run_policy)(const BBParams&, const BBParams& stage, const BBRunArgs&, const BBPolicy&,
                            unsigned long long counter0, int nwarps, cudaStream_t);
  int (*run_policy_warps_per_sm)(const BBParams&, int hidden);
};

const BBKernelTable* bb_kernel_table(int nvars);  // bbenv.cu; NULL if nvars is outside 1..8

#ifdef BB_NV  // ---------------------------------------------------------------------- per-NV translation unit only

// warp rows -> one global atomic per CTA and counter
__device__ __forceinline__ void counters_flush(const BBParams& P, unsigned long long (*sh)[CT_COUNT]) {
  __syncthreads();
  if (threadIdx.x < CT_COUNT) {
    unsigned long long s = 0;
#pragma unroll
    for (int w = 0; w < BB_WARPS; w++) s += sh[w][threadIdx.x];
    if (s) atomicAdd(&P.counters[threadIdx.x], s);
  }
}
__device__ __forceinline__ unsigned long long* counters_row(unsigned long long (*sh)[CT_COUNT]) {
  unsigned long long* row = sh[threadIdx.x >> 5];
  if (bb_lane() < CT_COUNT) row[bb_lane()] = 0ull;
  __syncwarp();
  return row;
}

// reset() of one environment of the step API: the head of its prefetch queue, else the generator (defined below)
template <int NV>
__device__ __noinline__ void warp_next_episode(const BBParams& P, int slot, unsigned long long* row);

template <int NV>
__global__ void __launch_bounds__(BB_THREADS, BB_MIN_BLOCKS) k_reset(const __grid_constant__ BBParams P, const uint8_t* mask) {
  __shared__ unsigned long long sh[BB_WARPS][CT_COUNT];
  hot_init(P);
  unsigned long long* row = counters_row(sh);
  const int slot = (blockIdx.x * BB_THREADS + threadIdx.x) >> 5;
  if (slot < P.num_envs && (!mask || mask[slot])) warp_next_episode<NV>(P, slot, row);
  counters_flush(P, sh);
}

// One environment step with the bookkeeping k_step and k_rollout share: per-slot episode record, counters, reward.
// Returns the reward (0 for a bad action).
template <int NV>
__device__ __forceinline__ double step_and_account(const BBParams& P, int slot, Env& e, int action, Ctr& ct,
                                                   unsigned long long* row) {
  uint32_t pr;
  const int g0 = e.nG;
  const int adds = warp_step<NV>(P, e, action, pr, ct);
  if (pr == 0xffffffffu) return 0.0;
  if (bb_lane() == 0) {
    const int pi = pr & 0xffffu, pj = pr >> 16;
    BBEnvState& S = P.st[slot];
    S.trace_hash = trace_hash_step(S.trace_hash, pr, adds);
    S.steps += 1; S.adds += adds;
    if (e.nG > g0) S.nonzero += 1; else S.zero += 1;
    row[CT_STEPS] += 1; row[CT_ADDS] += (unsigned)adds;
    row[e.nG > g0 ? CT_NONZERO : CT_ZERO] += 1;
    if (e.status == BB_STATUS_DONE) row[CT_EPISODES] += 1;
  }
  if (P.max_episode_length > 0 && e.status == BB_STATUS_RUNNING) {   // pg.py:470-471: cut once episode_length > max
    int n = 0;
    if (bb_lane() == 0) n = P.st[slot].steps;
    n = __shfl_sync(BB_FULL, n, 0);
    if (n > P.max_episode_length) {
      e.status = BB_STATUS_TRUNCATED;
      if (bb_lane() == 0) { P.st[slot].truncated = 1; row[CT_EPISODES] += 1; }
    }
  }
  return (P.rewards == BB_REWARD_ADDITIONS) ? -(double)adds : -1.0;
}

template <int NV>
__global__ void __launch_bounds__(BB_THREADS, BB_MIN_BLOCKS) k_step(const __grid_constant__ BBParams P,
                                                                   const int* __restrict__ actions,
                                                                   double* __restrict__ reward, uint8_t* __restrict__ done,
                                                                   const int* __restrict__ active) {
  __shared__ unsigned long long sh[BB_WARPS][CT_COUNT];
  hot_init(P);
  unsigned long long* row = counters_row(sh);
  const int w = (blockIdx.x * BB_THREADS + threadIdx.x) >> 5;
  // active (k_compact): warp w takes the w-th environment of the RUNNING-first order, so the stepping warps fill whole
  // CTAs and the CTAs behind them hold idle environments only
  const int slot = (active && w < P.num_envs) ? active[1 + w] : w;
  if (slot < P.num_envs) {
    Env e; env_load(P, slot, e);
    Ctr ct; ct.clear();
    double r = 0.0;
    if (e.status == BB_STATUS_RUNNING) {
      r = step_and_account<NV>(P, slot, e, actions[slot], ct, row);
      env_store(P, slot, e);
    }
    if (bb_lane() == 0) {
      if (reward) reward[slot] = r;
      if (done) done[slot] = (e.status != BB_STATUS_RUNNING) ? 1 : 0;
    }
    ct.spill(row);
    if (P.auto_reset && e.status != BB_STATUS_RUNNING) {  // the caller sees done = 1 and the NEXT episode's first state
      __syncwarp();
      warp_next_episode<NV>(P, slot, row);
    }
  }
  if (P.pre && blockIdx.x == 0 && threadIdx.x == 0) (*P.pre->calls)++;   // one step call more (see BBPre::calls)
  counters_flush(P, sh);
}

// step() as the reference's binding sees it (wrapped.pyx:23-26: step, then the state matrix and done, in ONE call):
// one launch does the step of every environment, the auto-reset if enabled, and the observation of the state AFTER it.
// `actions` may be NULL, then every environment takes `action0` (the single-environment drop-in passes its action by
// value: no host-to-device copy at all).  The outputs may be device memory or mapped pinned host memory.
// pad == 0: rows beyond |P| are left untouched (a host caller reads lengths first), else they are -1.
template <int NV>
__global__ void __launch_bounds__(BB_THREADS, BB_MIN_BLOCKS) k_step_obs(const __grid_constant__ BBParams P,
                                                                       const int* __restrict__ actions, int action0,
                                                                       double* __restrict__ reward, uint8_t* __restrict__ done,
                                                                       int32_t* __restrict__ obs, int32_t* __restrict__ lengths,
                                                                       int pmax, int pad, int do_step,
                                                                       const int* __restrict__ active,
                                                                       unsigned* __restrict__ ready, unsigned ticket) {
  __shared__ unsigned long long sh[BB_WARPS][CT_COUNT];
  hot_init(P);
  unsigned long long* row = counters_row(sh);
  const int w = (blockIdx.x * BB_THREADS + threadIdx.x) >> 5;
  const int slot = (active && w < P.num_envs) ? active[1 + w] : w;   // as k_step
  if (slot < P.num_envs) {
    Env e; env_load(P, slot, e);
    Ctr ct; ct.clear();
    if (do_step) {
      double r = 0.0;
      if (e.status == BB_STATUS_RUNNING) {
        r = step_and_account<NV>(P, slot, e, actions ? actions[slot] : action0, ct, row);
        env_store(P, slot, e);
      }
      if (bb_lane() == 0) {
        if (reward) reward[slot] = r;
        if (done) done[slot] = (e.status != BB_STATUS_RUNNING) ? 1 : 0;
      }
      if (P.auto_reset && e.status != BB_STATUS_RUNNING) {
        __syncwarp();
        warp_next_episode<NV>(P, slot, row);
        env_load(P, slot, e);
      }
    }
    if (obs) {
      const int rows = e.nP < pmax ? e.nP : pmax;
      warp_observe<NV>(P, e, obs + (size_t)slot * pmax * P.cols, pad ? pmax : rows, ct);
    }
    if (lengths && bb_lane() == 0) lengths[slot] = e.nP;
    ct.spill(row);
  }
  if (do_step && P.pre && blockIdx.x == 0 && threadIdx.x == 0) (*P.pre->calls)++;   // one step call more (see BBPre::calls)
  // single-CTA launches of bb_step_host: the results sit in mapped host memory; the host waits for this word instead of a
  // stream synchronisation (every thread's writes are made visible system-wide before thread 0 publishes the ticket)
  if (ready) __threadfence_system();
  counters_flush(P, sh);
  if (ready) {
    __syncthreads();
    if (threadIdx.x == 0) { *reinterpret_cast<volatile unsigned*>(ready) = ticket; __threadfence_system(); }
  }
}

// The single-environment server: ONE resident warp that executes reset() / step() / observe() of environment 0 on command,
// so that a host call of the reference's binding (wrapped.pyx:18-26: one environment, one action, the state matrix back)
// costs a PCIe round trip instead of a kernel launch and a stream synchronisation.  Same code as k_step_obs / k_reset.
// The warp leaves after idle_ns without a command (the host starts a new instance on demand), on BB_CMD_STOP, or with its
// environment's parameters changed (every other entry point of the library stops it first).
__device__ __forceinline__ unsigned long long bb_globaltimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
template <int NV>
__global__ void __launch_bounds__(32) k_serve(const __grid_constant__ BBParams P, BBMailbox* mb, unsigned long long idle_ns) {
  __shared__ unsigned long long sh[1][CT_COUNT];
  hot_init(P);
  const int lane = bb_lane();
  if (lane < CT_COUNT) sh[0][lane] = 0ull;
  __syncwarp();
  unsigned long long* row = sh[0];
  int32_t* obs = reinterpret_cast<int32_t*>(mb + 1);
  unsigned seen = mb->done_seq;
  unsigned long long t_idle = bb_globaltimer();
  for (;;) {
    uint4 c = make_uint4(0u, 0u, 0u, 0u);
    if (lane == 0)   // the host writes the 16 bytes with one aligned store: sequence number and command arrive together
      asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(c.x), "=r"(c.y), "=r"(c.z), "=r"(c.w) : "l"(mb));
    const unsigned s = __shfl_sync(BB_FULL, c.x, 0);
    if (s == seen) {
      if (bb_globaltimer() - t_idle > idle_ns) break;
      continue;
    }
    const unsigned cmd = __shfl_sync(BB_FULL, c.y, 0);
    const int arg = (int)__shfl_sync(BB_FULL, c.z, 0);
    const int rowsw = (int)__shfl_sync(BB_FULL, c.w, 0);
    const int pmax = rowsw >> 1, pad = rowsw & 1;
    if (cmd != BB_CMD_STOP) {
      Ctr ct; ct.clear();
      double r = 0.0;
      if (cmd == BB_CMD_RESET) warp_next_episode<NV>(P, 0, row);
      Env e; env_load(P, 0, e);
      if (cmd == BB_CMD_STEP) {
        if (e.status == BB_STATUS_RUNNING) {
          r = step_and_account<NV>(P, 0, e, arg, ct, row);
          env_store(P, 0, e);
        }
        if (lane == 0) { mb->reward = r; mb->done = (e.status != BB_STATUS_RUNNING) ? 1u : 0u; }
        if (P.auto_reset && e.status != BB_STATUS_RUNNING) {
          __syncwarp();
          warp_next_episode<NV>(P, 0, row);
          env_load(P, 0, e);
        }
      }
      if (pmax > 0) {
        const int rows = e.nP < pmax ? e.nP : pmax;
        warp_observe<NV>(P, e, obs, pad ? pmax : rows, ct);
      }
      if (lane == 0) mb->length = e.nP;
      ct.spill(row);
    }
    __threadfence_system();   // every lane's results before the sequence number
    __syncwarp();
    if (lane == 0) mb->done_seq = s;
    seen = s;
    if (cmd == BB_CMD_STOP) break;
    t_idle = bb_globaltimer();
  }
  __syncwarp();
  if (lane < CT_COUNT && sh[0][lane]) atomicAdd(&P.counters[lane], sh[0][lane]);
  __threadfence_system();
  __syncwarp();
  if (lane == 0) { mb->alive = 0u; __threadfence_system(); }
}

template <int NV>
__global__ void __launch_bounds__(BB_THREADS) k_select(const __grid_constant__ BBParams P, int strategy,
                                                       int* __restrict__ actions) {
  const int slot = (blockIdx.x * BB_THREADS + threadIdx.x) >> 5;
  if (slot >= P.num_envs) return;
  Env e; env_load(P, slot, e);
  const int a = (e.status == BB_STATUS_RUNNING) ? warp_select<NV>(P, e, strategy, &P.st[slot].sel_rng) : 0;
  if (bb_lane() == 0) actions[slot] = a;
}

template <int NV>
__global__ void __launch_bounds__(BB_THREADS) k_observe(const __grid_constant__ BBParams P, int32_t* __restrict__ obs,
                                                        int32_t* __restrict__ lengths, int pmax) {
  __shared__ unsigned long long sh[BB_WARPS][CT_COUNT];
  unsigned long long* row = counters_row(sh);
  const int slot = (blockIdx.x * BB_THREADS + threadIdx.x) >> 5;
  if (slot < P.num_envs) {
    Env e; env_load(P, slot, e);
    Ctr ct; ct.clear();
    if (obs) warp_observe<NV>(P, e, obs + (size_t)slot * pmax * P.cols, pmax, ct);
    if (lengths && bb_lane() == 0) lengths[slot] = e.nP;
    ct.spill(row);
  }
  counters_flush(P, sh);
}

template <int NV>
__global__ void __launch_bounds__(32) k_final_gb(const __grid_constant__ BBParams P, int slot, int* ok_out) {
  __shared__ unsigned long long sh[1][CT_COUNT];
  if (bb_lane() < CT_COUNT) sh[0][bb_lane()] = 0ull;
  __syncwarp();
  const int ok = warp_final_gb<NV>(P, slot, sh[0]);
  if (bb_lane() == 0) *ok_out = ok;
}

// Episode preparation: warp b of the batch draws episode (ep_base + b)'s ideal from its stream and runs
// BuchbergerEnv::reset on it (re-rolls included) inside the compact staging arena S (one small slot per episode of
// the batch).  Keeping this out of k_run keeps the generator / reset code out of the step loop's instruction
// working set (profiles/r01_v2: instruction fetch was the top stall) and runs it with every warp in the same code.
template <int NV>
__global__ void __launch_bounds__(BB_THREADS, BB_MIN_BLOCKS) k_prepare(const __grid_constant__ BBParams S,
                                                                      const __grid_constant__ BBRunArgs A) {
  __shared__ unsigned long long sh[BB_WARPS][CT_COUNT];
  hot_init(S);
  unsigned long long* row = counters_row(sh);
  const int b = (blockIdx.x * BB_THREADS + threadIdx.x) >> 5;
  if (b < A.episodes) {
    const int ep = A.ep_base + b;
    warp_reset_slot<NV>(S, b, S.dist.enabled ? b : (A.ep_offset + ep) % A.nstaged, rng_seed(A.seeds ? A.seeds[ep] : A.seed_base + ep), row);
    // Predicted cost of the episode, for the longest-first queue order: the summed degree of the generators' lead
    // monomials (rank correlation with the episode length ~0.5 on the binomial distributions), scaled to a bucket.
    // Only the ORDER in which episodes start depends on it, never a result.
    const int nG = S.st[b].nG;
    const uint64_t* lm = SLOT_PTR(uint64_t, S, b, o_lm);
    uint32_t sd = 0;
    for (int i = bb_lane(); i < nG; i += 32) sd += KL<NV>::deg(lm[i]);
    sd = __reduce_add_sync(BB_FULL, sd);
    if (bb_lane() == 0) {
      // generated ideals: s generators of degree <= d; a fixed ideal is the same for every episode (one bucket)
      uint32_t key = S.dist.enabled ? (sd * (BB_LPT_BUCKETS - 1)) / (uint32_t)max(1, S.dist.s * S.dist.d) : 0u;
      key = key < BB_LPT_BUCKETS ? key : BB_LPT_BUCKETS - 1;
      A.cost_key[b] = (uint8_t)key;
      atomicAdd(&A.queue[BB_LPT_HIST + key], 1);
    }
  }
  counters_flush(S, sh);
}

// The same preparation with ONE THREAD per episode, for the binomial distributions (RandomBinomialIdealGenerator,
// ideals.cpp:168-201) with at most BB_PREP_S generators: the generator and the s update() calls of reset()
// (buchberger.cpp:299-315, :52-99) are a few thousand scalar instructions on <= 16 lead monomials and <= 120 pairs, so
// a warp that spends them on one episode (k_prepare) wastes 31 lanes; here a warp prepares 32 episodes in lockstep
// out of thread-local arrays and writes each finished state to its staging slot.  Same results, same counters.
// update() in closed form (see warp_add_basis): with L_i = lcm(LM_i, LM f), (i, m) is emitted iff no L_j strictly divides
// L_i, no j < i has L_j == L_i, and no j with L_j == L_i is coprime to f.
#define BB_PREP_P (BB_PREP_S * (BB_PREP_S - 1) / 2)
#ifndef BB_PREP_THREADS
#define BB_PREP_THREADS 32
#endif
#ifndef BB_PREP_MIN_BLOCKS
#define BB_PREP_MIN_BLOCKS 1
#endif
// One episode prepared by ONE thread: the ideal drawn from the stream state x (advanced), BuchbergerEnv::reset on it (re-rolls
// included), the finished state written to slot b of the staging arena S.  Returns the summed degree of the generators' lead
// monomials (the episode's predicted cost); upb / upp accumulate the update() traffic counters.
template <int NV>
__device__ __forceinline__ uint32_t prepare_lane_episode(const BBParams& S, int b, uint32_t& x, unsigned& upb, unsigned& upp) {
  typedef KL<NV> K;
  const BBDist& D = S.dist;
  const BBField F = S.F;
  const int s = D.s;
  uint64_t gk0[BB_PREP_S], gk1[BB_PREP_S];          // generators: lead / second monomial, second coefficient (lead coefficient 1)
  uint32_t gc1[BB_PREP_S];
  uint64_t L[BB_PREP_S];                             // update(): key of lcm(LM_i, LM f)
  uint64_t rl[BB_PREP_S]; uint32_t ri[BB_PREP_S];    // reducer list G_
  uint32_t prs[BB_PREP_P]; uint64_t plc[BB_PREP_P];  // pair list P with cached lcm keys
  int nG = 0, nP = 0, status = BB_STATUS_EMPTY, rerolls = 0;
  for (;;) {
    bool ok = true;
    for (int i = 0; i < s && ok; i++) {   // RandomBinomialIdealGenerator::next, as gen_binomial_ideal
      const uint32_t c = D.pure ? (F.p - 1u) : (uint32_t)rng_uniform(x, 1, (int)F.p - 1);
      int d1, d2;
      if (D.homogeneous) d1 = d2 = rng_degree(D, x);
      else { d1 = rng_degree(D, x); d2 = rng_degree(D, x); }
      const int o1 = D.basis_off[d1], n1 = D.basis_off[d1 + 1] - o1, o2 = D.basis_off[d2], n2 = D.basis_off[d2 + 1] - o2;
      ok = false;
      for (int trials = 0; trials < 1000 && !ok; trials++) {
        const uint64_t m1 = D.basis[o1 + rng_uniform(x, 0, n1 - 1)];
        const uint64_t m2 = D.basis[o2 + rng_uniform(x, 0, n2 - 1)];
        if (m1 != m2) { gk0[i] = m1 < m2 ? m1 : m2; gk1[i] = m1 < m2 ? m2 : m1; gc1[i] = c; ok = true; }
      }
    }
    if (!ok) { nG = nP = 0; status = BB_STATUS_EMPTY; break; }   // the reference throws (ideals.cpp:196-197)
    if (S.sort_input) {   // ascending lead monomial == descending key, stable (buchberger.cpp:301-302; see warp_load_ideal)
      for (int i = 1; i < s; i++) {
        const uint64_t a0 = gk0[i], a1 = gk1[i]; const uint32_t ac = gc1[i];
        int j = i;
        while (j > 0 && gk0[j - 1] < a0) { gk0[j] = gk0[j - 1]; gk1[j] = gk1[j - 1]; gc1[j] = gc1[j - 1]; j--; }
        gk0[j] = a0; gk1[j] = a1; gc1[j] = ac;
      }
    }
    nG = 0; nP = 0; status = BB_STATUS_RUNNING;
    for (int m = 0; m < s; m++) {   // update(G, P, f) + insertion into G_, generator by generator
      const uint64_t fk = gk0[m], fe = fk & K::ex_mask;
      upb += (unsigned)m; upp += (unsigned)nP;
      int kept = nP;   // old pairs that survive
      if (S.elimination == BB_ELIM_GEBAUERMOELLER) {
        bool ovf = false;
        uint32_t cop = 0u;
        for (int i = 0; i < m; i++) {
          const uint64_t le = K::lcm_exps(gk0[i], fk);
          const uint32_t dg = K::sum_fields(le);
          ovf |= dg > K::dmax;
          L[i] = le | ((uint64_t)(K::dmax - dg) << K::dshift);
          cop |= K::coprime(gk0[i], fk) ? (1u << i) : 0u;
        }
        if (ovf) { status = BB_STATUS_OVERFLOW_EXPONENT; break; }
        int w = 0;
        for (int q = 0; q < nP; q++) {
          const uint32_t pr = prs[q]; const uint64_t pl = plc[q];
          const uint64_t l = pl & K::ex_mask;
          const bool drop = K::divides(fe, l) && l != (L[pr & 0xffffu] & K::ex_mask) && l != (L[pr >> 16] & K::ex_mask);
          if (!drop) { prs[w] = pr; plc[w] = pl; w++; }
        }
        nP = w; kept = w;
        for (int i = 0; i < m; i++) {
          const uint64_t li = L[i] & K::ex_mask;
          bool emit = true;
          for (int j = 0; j < m && emit; j++) {   // a third of this kernel's instructions were spent here without the early exit
            const uint64_t lj = L[j] & K::ex_mask;
            if (lj == li) emit = emit && !(j < i) && !((cop >> j) & 1u);
            else emit = emit && !((((li | K::ge_mask) - lj) & K::ge_mask) == K::ge_mask);
          }
          if (emit) { prs[nP] = ((uint32_t)m << 16) | (uint32_t)i; plc[nP] = L[i]; nP++; }
        }
      } else {
        for (int i = 0; i < m; i++) {
          if (S.elimination == BB_ELIM_LCM && K::coprime(gk0[i], fk)) continue;
          prs[nP] = ((uint32_t)m << 16) | (uint32_t)i; plc[nP] = K::key_from_exps(K::lcm_exps(gk0[i], fk)); nP++;
        }
      }
      upp += (unsigned)(nP - kept);   // emitted pairs, counted as warp_load_ideal counts them
      int pos = m;
      if (S.sort_reducers) {   // after every element whose lead monomial is <= the new one (key >= new key)
        pos = 0;
        while (pos < m && rl[pos] >= fk) pos++;
        for (int r = m; r > pos; r--) { rl[r] = rl[r - 1]; ri[r] = ri[r - 1]; }
      }
      rl[pos] = fk; ri[pos] = (uint32_t)m;
      nG = m + 1;
    }
    if (status != BB_STATUS_RUNNING || nP > 0) break;
    rerolls++;   // P came out empty: the next ideal of the same stream (buchberger.cpp:313-314)
  }
  if (status == BB_STATUS_RUNNING && nP == 0) status = BB_STATUS_DONE;
  // the finished state goes to the episode's staging slot
  unsigned char* base = S.arena + (size_t)b * S.slot_stride;
  GHeadMem* gh = reinterpret_cast<GHeadMem*>(base + S.o_ghead);
  uint64_t* lm = reinterpret_cast<uint64_t*>(base + S.o_lm);
  uint64_t* rlm = reinterpret_cast<uint64_t*>(base + S.o_rlm);
  uint32_t* ridx = reinterpret_cast<uint32_t*>(base + S.o_ridx);
  uint32_t* pairs = reinterpret_cast<uint32_t*>(base + S.o_pairs);
  uint64_t* plcm = reinterpret_cast<uint64_t*>(base + S.o_plcm);
  uint64_t* tk = reinterpret_cast<uint64_t*>(base + S.o_tkey);
  uint32_t* tc = reinterpret_cast<uint32_t*>(base + S.o_tcoef);
  uint32_t sd = 0;
  for (int m = 0; m < nG; m++) {
    const uint64_t fk = gk0[m], k1 = gk1[m];
    reinterpret_cast<uint4*>(gh + m)[0] = make_uint4((uint32_t)fk, (uint32_t)(fk >> 32), (uint32_t)k1, (uint32_t)(k1 >> 32));
    reinterpret_cast<uint4*>(gh + m)[1] = make_uint4(1u | (gc1[m] << 16), K::deg(fk), (uint32_t)(2 * m), 2u);   // 1 / LC = 1
    lm[m] = fk; rlm[m] = rl[m]; ridx[m] = ri[m];
    tk[2 * m] = fk; tk[2 * m + 1] = k1; tc[2 * m] = 1u; tc[2 * m + 1] = gc1[m];
    sd += K::deg(fk);
  }
  for (int q = 0; q < nP; q++) { pairs[q] = prs[q]; plcm[q] = plc[q]; }
  *reinterpret_cast<int4*>(&S.st[b]) = make_int4(nG, nP, 2 * nG, status);
  S.st[b].rng = x; S.st[b].rerolls = rerolls;
  return sd;
}

template <int NV>
__global__ void __launch_bounds__(BB_PREP_THREADS, BB_PREP_MIN_BLOCKS) k_prepare_lanes(const __grid_constant__ BBParams S,
                                                                    const __grid_constant__ BBRunArgs A) {
  __shared__ unsigned long long sh_up[2];
  if (threadIdx.x < 2) sh_up[threadIdx.x] = 0ull;
  __syncthreads();
  const int b = blockIdx.x * BB_PREP_THREADS + threadIdx.x;
  unsigned upb = 0u, upp = 0u;
  if (b < A.episodes) {
    const int ep = A.ep_base + b;
    uint32_t x = rng_seed(A.seeds ? A.seeds[ep] : A.seed_base + ep);
    const uint32_t sd = prepare_lane_episode<NV>(S, b, x, upb, upp);
    uint32_t key = (sd * (BB_LPT_BUCKETS - 1)) / (uint32_t)max(1, S.dist.s * S.dist.d);
    key = key < BB_LPT_BUCKETS ? key : BB_LPT_BUCKETS - 1;
    A.cost_key[b] = (uint8_t)key;
    atomicAdd(&A.queue[BB_LPT_HIST + key], 1);
  }
  upb = __reduce_add_sync(BB_FULL, upb); upp = __reduce_add_sync(BB_FULL, upp);
  if (bb_lane() == 0) { atomicAdd(&sh_up[0], (unsigned long long)upb); atomicAdd(&sh_up[1], (unsigned long long)upp); }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (sh_up[0]) atomicAdd(&S.counters[CT_UPB], sh_up[0]);
    if (sh_up[1]) atomicAdd(&S.counters[CT_UPP], sh_up[1]);
  }
}

// Queue order of a batch: episodes sorted by cost bucket, largest first (counting sort).  Every CTA recomputes the
// bucket starts from the histogram and places a slice of the batch through the global per-bucket cursors.  Within a
// bucket the order is whatever the atomics produce -- it only decides which worker warp picks an episode up when.
template <int NV>
__global__ void __launch_bounds__(BB_LPT_BUCKETS) k_order(const __grid_constant__ BBRunArgs A) {
  __shared__ int hist[BB_LPT_BUCKETS], start[BB_LPT_BUCKETS];
  const int t = threadIdx.x;
  hist[t] = A.queue[BB_LPT_HIST + t];
  __syncthreads();
  int before = 0;
  for (int k = t + 1; k < BB_LPT_BUCKETS; k++) before += hist[k];
  start[t] = before;
  __syncthreads();
  int* cursor = A.queue + BB_LPT_HIST + BB_LPT_BUCKETS;
  for (int b = blockIdx.x * BB_LPT_BUCKETS + t; b < A.episodes; b += gridDim.x * BB_LPT_BUCKETS) {
    const int key = A.cost_key[b];
    A.order[start[key] + atomicAdd(&cursor[key], 1)] = b;
  }
}

// copy n 32-bit words, lane-strided
__device__ __forceinline__ void warp_copy_words(uint32_t* __restrict__ d, const uint32_t* __restrict__ s, int n) {
  d = bb_global(d); s = bb_global(s);
#pragma unroll 1
  for (int t = bb_lane(); t < n; t += 32) d[t] = s[t];
}

// copy the live part of environment `src` (arena base sb, scalars in e) into the arena at db (same layout)
__device__ __forceinline__ void warp_copy_env(const BBParams& D, unsigned char* db, const BBParams& S, const unsigned char* sb,
                                              const Env& e) {
  warp_copy_words((uint32_t*)(db + D.o_ghead), (const uint32_t*)(sb + S.o_ghead), e.nG * 8);
  warp_copy_words((uint32_t*)(db + D.o_lm), (const uint32_t*)(sb + S.o_lm), e.nG * 2);
  warp_copy_words((uint32_t*)(db + D.o_rlm), (const uint32_t*)(sb + S.o_rlm), e.nG * 2);
  warp_copy_words((uint32_t*)(db + D.o_ridx), (const uint32_t*)(sb + S.o_ridx), e.nG);
  warp_copy_words((uint32_t*)(db + D.o_pairs), (const uint32_t*)(sb + S.o_pairs), e.nP);
  warp_copy_words((uint32_t*)(db + D.o_plcm), (const uint32_t*)(sb + S.o_plcm), e.nP * 2);
  warp_copy_words((uint32_t*)(db + D.o_tkey), (const uint32_t*)(sb + S.o_tkey), e.nT * 2);
  warp_copy_words((uint32_t*)(db + D.o_tcoef), (const uint32_t*)(sb + S.o_tcoef), e.nT);
}

template <int NV>
__device__ __noinline__ void warp_next_episode(const BBParams& P, int slot, unsigned long long* row) {
  const int lane = bb_lane();
  const BBPre* Q = P.pre;
  if (Q && P.dist.enabled) {
    const int cnt = Q->count[slot], hd = Q->head[slot], depth = Q->depth;
    __syncwarp();   // every lane has read the queue words before lane 0 moves them
    if (cnt > 0) {
      const int idx = slot * depth + hd;
      Env se; env_load(Q->S, idx, se);
      unsigned char* db = bb_global(P.arena + (size_t)slot * P.slot_stride);
      warp_copy_env(P, db, Q->S, se.base, se);
      __syncwarp();
      if (lane == 0) {
        BBEnvState& T = P.st[slot];
        const BBEnvState& U = Q->S.st[idx];
        *reinterpret_cast<int4*>(&T) = make_int4(se.nG, se.nP, se.nT, se.status);
        T.rng = U.rng; T.rerolls = U.rerolls;
        T.steps = 0; T.adds = 0; T.zero = 0; T.nonzero = 0; T.truncated = 0;
        T.trace_hash = 0; T.disc_return = 0.0; T.discount = 1.0;
        Q->head[slot] = hd + 1 == depth ? 0 : hd + 1;
        Q->count[slot] = cnt - 1;
      }
      __syncwarp();
      return;
    }
  }
  warp_reset_slot<NV>(P, slot, slot, (uint32_t)P.st[slot].rng, row);
  if (Q && P.dist.enabled && lane == 0) Q->rng[slot] = (uint32_t)P.st[slot].rng;   // empty queue: its tail is the new position
  __syncwarp();
}

// Tops the prefetch queues up: thread e prepares the next episodes of environment e's stream until its queue is full.
template <int NV>
__global__ void __launch_bounds__(BB_PREP_THREADS, BB_PREP_MIN_BLOCKS) k_prefill(const __grid_constant__ BBParams P,
                                                                               const __grid_constant__ BBParams S, int period) {
  if (period > 0 && (*P.pre->calls % period) != 0) return;   // nobody writes the counter while this kernel runs
  __shared__ unsigned long long sh_up[2];
  if (threadIdx.x < 2) sh_up[threadIdx.x] = 0ull;
  __syncthreads();
  const int e = blockIdx.x * BB_PREP_THREADS + threadIdx.x;
  unsigned upb = 0u, upp = 0u;
  const BBPre* Q = P.pre;
  if (e < P.num_envs) {
    const int depth = Q->depth;
    int cnt = Q->count[e];
    if (cnt < depth) {
      uint32_t x = Q->rng[e];
      int tail = Q->head[e] + cnt;
      if (tail >= depth) tail -= depth;
      while (cnt < depth) {
        prepare_lane_episode<NV>(S, e * depth + tail, x, upb, upp);
        tail = tail + 1 == depth ? 0 : tail + 1;
        cnt++;
      }
      Q->count[e] = cnt;
      Q->rng[e] = x;
    }
  }
  upb = __reduce_add_sync(BB_FULL, upb); upp = __reduce_add_sync(BB_FULL, upp);
  if (bb_lane() == 0) { atomicAdd(&sh_up[0], (unsigned long long)upb); atomicAdd(&sh_up[1], (unsigned long long)upp); }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (sh_up[0]) atomicAdd(&P.counters[CT_UPB], sh_up[0]);
    if (sh_up[1]) atomicAdd(&P.counters[CT_UPP], sh_up[1]);
  }
}

// The loop of buchberger() (buchberger.cpp:243-263) on one environment: select, step, accumulate the trace checksum and
// the discounted return (discounted_return += discount * reward; discount *= gamma, :250-251) until P is empty.
// TWO: see warp_step.  UPL > 0: the pairs policy head (bb_policy.cuh, H = 32 * UPL, weights at wsm) selects instead of
// `strategy`; step t draws its uniform from (W->seed + stream, counter0 + t), stream = the episode's global index.
template <int NV, bool TWO = false, int UPL = 0>
__device__ __forceinline__ void run_episode(const BBParams& P, Env& e, int strategy, int max_steps, double gamma,
                                            BBEpisodeAcc& acc, Ctr& ct, int& steps, int& adds, int4* trace, int trace_cap,
                                            const BBPolicy* W = nullptr, const float* wsm = nullptr,
                                            unsigned long long stream = 0, unsigned long long counter0 = 0) {
  const int lane = bb_lane();
  while (e.status == BB_STATUS_RUNNING && (max_steps == 0 || steps < max_steps)) {
    int prow;
    if constexpr (UPL > 0) {
      float lp;
      prow = warp_policy<NV, UPL>(P, e, wsm, W->greedy, policy_uniform(W->seed, stream, counter0 + (unsigned)steps), lp,
                                  nullptr, 0);
    } else {
      prow = warp_select<NV>(P, e, strategy, &acc.sel_rng);
    }
    uint32_t pr;
    const int a = warp_step<NV, TWO>(P, e, prow, pr, ct);
    if (lane == 0) {
      const int pi = pr & 0xffffu, pj = pr >> 16;
      acc.th = trace_hash_step(acc.th, pr, a);
      const double r = (P.rewards == BB_REWARD_ADDITIONS) ? -(double)a : -1.0;
      const double d = acc.disc;
      acc.ret = __dadd_rn(acc.ret, __dmul_rn(d, r)); acc.disc = __dmul_rn(d, gamma);
      if (trace && steps < trace_cap) trace[steps] = make_int4(pi, pj, a, e.nP);
    }
    steps++; adds += a;
  }
}

// bb_run_export's sinks at the end of episode `ep` of slot `slot` (the runners' epilogue, after env_store and the reduced
// basis): the reduced basis of an episode that ends done from the slot's GB arena, G of an episode that ends done or is cut
// by max_steps (status still running) from the slot's term arena.  One out-of-line call per episode, and only when a sink
// is attached, so the runners' step loop does not change.
template <int NV>
__device__ __noinline__ void warp_export_episode(const BBParams& P, const BBRunArgs& A, int slot, int ep, int status) {
  if (A.gb_sink.lens_dev && status == BB_STATUS_DONE)
    warp_export_polys<NV>(P.gkey + (size_t)slot * P.max_terms, P.gcoef + (size_t)slot * P.max_terms,
                          P.glen + (size_t)slot * P.max_basis, 1, P.gcount[2 * slot], P.gcount[2 * slot + 1], A.gb_sink, ep);
  if (A.basis_sink.lens_dev && (status == BB_STATUS_DONE || status == BB_STATUS_RUNNING)) {
    Env e; env_load(P, slot, e);
    const GHeadMem* gh = ENV_PTR(GHeadMem, e, P, o_ghead);
    warp_export_polys<NV>(ENV_PTR(uint64_t, e, P, o_tkey), ENV_PTR(uint32_t, e, P, o_tcoef),
                          reinterpret_cast<const int*>(&gh[0].len), (int)(sizeof(GHeadMem) / sizeof(int)), e.nG, e.nT,
                          A.basis_sink, ep);
  }
}

// Persistent episode runner.  Each warp owns slot = its global warp index and loops: pop an episode, copy its
// prepared initial state from the staging arena, select/step until P is empty (or max_steps), write the episode
// record, repeat.  WARPS = warps per CTA.  EXPORT: bb_run_export's sinks may be attached (an instantiation of its own, so
// the runner without sinks keeps the parent's code: k_run is issue- and instruction-footprint-bound, and the one extra call
// site in its loop measured 3 % on configs[1]).  TWO: the two-term step (warp_step), for runs whose ideals are binomial.
// UPL > 0: the policy head selects (run_episode; W, wsm: the weights and their shared-memory image, counter0: the counter
// of step 0).
template <int NV, int WARPS, bool EXPORT, bool TWO = false, int UPL = 0>
__device__ __forceinline__ void run_worker(const BBParams& P, const BBParams& S, const BBRunArgs& A,
                                           const BBPolicy* W = nullptr, const float* wsm = nullptr,
                                           unsigned long long counter0 = 0) {
  __shared__ unsigned long long sh[WARPS][CT_COUNT];
  __shared__ BBEpisodeAcc acc_sh[WARPS];  // per-episode accumulators only lane 0 touches: kept out of registers
  hot_init(P);
  unsigned long long* row = sh[threadIdx.x >> 5];
  if (bb_lane() < CT_COUNT) row[bb_lane()] = 0ull;
  __syncwarp();
  BBEpisodeAcc& acc = acc_sh[threadIdx.x >> 5];
  const int slot = (blockIdx.x * (WARPS * 32) + threadIdx.x) >> 5;
  const int lane = bb_lane();
  if (slot < P.num_envs) {
    Ctr ct; ct.clear();
    for (;;) {
      int b = 0;
      if (lane == 0) { b = atomicAdd(bb_global(A.queue), 1); b = b < A.episodes ? bb_global(A.order)[b] : -1; }
      b = __shfl_sync(BB_FULL, b, 0);
      if (b < 0) break;
      const int ep = A.ep_base + b;
      Env e; env_load(S, b, e);  // the prepared state; e.base still points into the staging arena here
      {
        unsigned char* db = bb_global(P.arena + (size_t)slot * P.slot_stride);
        warp_copy_env(P, db, S, e.base, e);
        e.base = db;
        __syncwarp();
      }
      const int g_start = e.nG;
      int steps = 0, adds = 0;
      if (lane == 0) { acc.th = 0ull; acc.ret = 0.0; acc.disc = 1.0; acc.sel_rng = rng_seed(A.sel_seed_base + (A.ep_offset + ep) * A.sel_seed_stride); }
      __syncwarp();
      run_episode<NV, TWO, UPL>(P, e, A.strategy, A.max_steps, A.gamma, acc, ct, steps, adds,
                               (A.trace && ep < A.trace_eps) ? reinterpret_cast<int4*>(A.trace) + (size_t)ep * A.trace_cap : nullptr,
                               A.trace_cap, W, wsm, (unsigned long long)(A.ep_offset + ep), counter0);
      const int nonzero = e.nG - g_start, zero = steps - nonzero;
      env_store(P, slot, e);
      __syncwarp();
      const GHeadMem* gh = ENV_PTR(GHeadMem, e, P, o_ghead);
      const unsigned long long bh = warp_terms_hash<NV>(ENV_PTR(uint64_t, e, P, o_tkey), ENV_PTR(uint32_t, e, P, o_tcoef),
                                                        e.nT, reinterpret_cast<const int*>(&gh[0].len),
                                                        (int)(sizeof(GHeadMem) / sizeof(int)), e.nG);
      unsigned long long gbh = 0; int gp = 0, gt = 0;
      int status = e.status;
      if (A.compute_gb && status == BB_STATUS_DONE) {
        if (warp_final_gb<NV>(P, slot, row)) {
          gp = P.gcount[2 * slot]; gt = P.gcount[2 * slot + 1];
          gbh = warp_terms_hash<NV>(P.gkey + (size_t)slot * P.max_terms, P.gcoef + (size_t)slot * P.max_terms, gt,
                                    P.glen + (size_t)slot * P.max_basis, 1, gp);
        } else {
          status = BB_STATUS_OVERFLOW_SCRATCH;
        }
      }
      if (EXPORT && (A.gb_sink.lens_dev || A.basis_sink.lens_dev)) warp_export_episode<NV>(P, A, slot, ep, status);
      if (lane == 0) {
        const unsigned long long th = acc.th; const double ret = acc.ret;
        bb_episode_stats o;
        o.steps = steps; o.additions = adds; o.zero_reductions = zero; o.nonzero_reductions = nonzero;
        o.nbasis = e.nG; o.nterms = e.nT; o.status = status; o.rerolls = S.st[b].rerolls;
        o.trace_hash = th; o.basis_hash = bh; o.gb_hash = gbh; o.gb_polys = gp; o.gb_terms = gt;
        o.discounted_return = ret;
        A.out[ep] = o;
        BBEnvState& St = P.st[slot];
        St.status = status; St.steps = steps; St.adds = adds; St.zero = zero; St.nonzero = nonzero; St.trace_hash = th;
        St.disc_return = ret; St.rerolls = o.rerolls;
        row[CT_STEPS] += (unsigned)steps; row[CT_ADDS] += (unsigned)adds; row[CT_NONZERO] += (unsigned)nonzero;
        row[CT_ZERO] += (unsigned)zero; row[CT_EPISODES] += 1;
      }
      ct.spill(row);
      __syncwarp();
    }
  }
  __syncthreads();
  if (threadIdx.x < CT_COUNT) {
    unsigned long long s = 0;
#pragma unroll
    for (int w = 0; w < WARPS; w++) s += sh[w][threadIdx.x];
    if (s) atomicAdd(&P.counters[threadIdx.x], s);
  }
}

template <int NV, bool EXPORT = false, bool TWO = false>
__global__ void __launch_bounds__(TWO ? BB_TWO_WARPS * 32 : BB_THREADS, TWO ? BB_TWO_MIN_BLOCKS : BB_MIN_BLOCKS)
k_run(const __grid_constant__ BBParams P, const __grid_constant__ BBParams S, const __grid_constant__ BBRunArgs A) {
  run_worker<NV, TWO ? BB_TWO_WARPS : BB_WARPS, EXPORT, TWO>(P, S, A);
}

// The same runner with the pairs policy head choosing the pairs (bb_run_policy): k_rollout's head and step (the general
// materialising warp_step for every ideal) in k_run's loop, so k_rollout's launch bounds.  The weight image lives in dynamic
// shared memory; policy_load_weights synchronises the CTA, so it comes before any slot check.  The sinks are checked at run
// time (an episode here is dominated by the head, not by the epilogue's call site).
template <int NV, int UPL>
__global__ void __launch_bounds__(BB_THREADS, BB_ROLLOUT_MIN_BLOCKS)
k_run_policy(const __grid_constant__ BBParams P, const __grid_constant__ BBParams S, const __grid_constant__ BBRunArgs A,
             const __grid_constant__ BBPolicy W, unsigned long long counter0) {
  extern __shared__ float wsm[];
  policy_load_weights(W, P.cols, wsm);
  run_worker<NV, BB_WARPS, true, false, UPL>(P, S, A, &W, wsm, counter0);
}

// block-strided copy of n 32-bit words
__device__ __forceinline__ void block_copy_words(uint32_t* __restrict__ d, const uint32_t* __restrict__ s, int n) {
  d = bb_global(d); s = bb_global(s);
#pragma unroll 1
  for (int t = threadIdx.x; t < n; t += BBW_THREADS) d[t] = s[t];
}

// Persistent episode runner, one CTA per environment slot (bb_wide.cuh): same queue, staging arena, episode record and
// checksums as k_run; the step is block_step.  Dynamic shared memory: the streams beyond one per thread.
template <int NV>
__global__ void __launch_bounds__(BBW_THREADS, BBW_MIN_CTAS) k_run_wide(const __grid_constant__ BBParams P, const __grid_constant__ BBParams S,
                                                          const __grid_constant__ BBRunArgs A) {
  extern __shared__ __align__(16) unsigned char wide_smem[];
  __shared__ unsigned long long sh[1][CT_COUNT];
  __shared__ BBEpisodeAcc acc;
  __shared__ WideShared wsh;
  __shared__ int next_b;
  WideStreams& st = *reinterpret_cast<WideStreams*>(wide_smem);   // streams beyond one per thread (bb_wide.cuh)
  const int tid = threadIdx.x;
  const int slot = blockIdx.x;
  hot_init(P);
  if (tid < CT_COUNT) sh[0][tid] = 0ull;
  __syncthreads();
  unsigned long long* row = sh[0];
  Ctr ct; ct.clear();
  WideState ws;
  ws.clear(); ws.cz = 0;
#ifdef BBW_INSTR
  ws.n_rounds = ws.n_trounds = ws.sum_T = ws.n_consol = ws.n_crounds = ws.n_topen = 0;
#endif
#ifdef BBW_CLOCK
  ws.cw = ws.cb = ws.cp = ws.co = ws.s_sel = ws.s_take = ws.s_red = ws.s_upd = 0; ws.tl = clock64();
#endif
  ws.regs = A.stream_regs < BBW_SLOTS ? (A.stream_regs < 2 ? 2 : A.stream_regs) : BBW_SLOTS;
  ws.cbase = A.ctl_reducers >= 32 && A.ctl_reducers < 256 ? (A.ctl_reducers & ~31) : 256;
  ws.tcap = A.stream_kmax - ws.regs < 0 ? 0 : (A.stream_kmax - ws.regs < BBW_KMAX - BBW_THREADS ? A.stream_kmax - ws.regs : BBW_KMAX - BBW_THREADS);
  int half = 0;
  for (;;) {
    if (tid == 0) { int q = atomicAdd(A.queue, 1); next_b = q < A.episodes ? A.order[q] : -1; }
    __syncthreads();
    const int b = next_b;
    if (b < 0) break;
    const int ep = A.ep_base + b;
    Env e; env_load(S, b, e);
    {
      unsigned char* db = P.arena + (size_t)slot * P.slot_stride;
      const unsigned char* sb = e.base;
      block_copy_words((uint32_t*)(db + P.o_ghead), (const uint32_t*)(sb + S.o_ghead), e.nG * 8);
      block_copy_words((uint32_t*)(db + P.o_lm), (const uint32_t*)(sb + S.o_lm), e.nG * 2);
      block_copy_words((uint32_t*)(db + P.o_rlm), (const uint32_t*)(sb + S.o_rlm), e.nG * 2);
      block_copy_words((uint32_t*)(db + P.o_ridx), (const uint32_t*)(sb + S.o_ridx), e.nG);
      block_copy_words((uint32_t*)(db + P.o_pairs), (const uint32_t*)(sb + S.o_pairs), e.nP);
      block_copy_words((uint32_t*)(db + P.o_plcm), (const uint32_t*)(sb + S.o_plcm), e.nP * 2);
      block_copy_words((uint32_t*)(db + P.o_tkey), (const uint32_t*)(sb + S.o_tkey), e.nT * 2);
      block_copy_words((uint32_t*)(db + P.o_tcoef), (const uint32_t*)(sb + S.o_tcoef), e.nT);
      e.base = db;
    }
    const int g_start = e.nG;
    int steps = 0, adds = 0;
    if (tid == 0) { acc.th = 0ull; acc.ret = 0.0; acc.disc = 1.0; acc.sel_rng = rng_seed(A.sel_seed_base + (A.ep_offset + ep) * A.sel_seed_stride); }
    __syncthreads();
    int4* trace = (A.trace && ep < A.trace_eps) ? reinterpret_cast<int4*>(A.trace) + (size_t)ep * A.trace_cap : nullptr;
    while (e.status == BB_STATUS_RUNNING && (A.max_steps == 0 || steps < A.max_steps)) {
      uint32_t pr;
      const int a = block_step<NV>(P, e, wsh, half, ws, st, A.strategy, &acc.sel_rng, pr, ct);
      if (tid == 0) {
        const int pi = pr & 0xffffu, pj = pr >> 16;
        acc.th = trace_hash_step(acc.th, pr, a);
        const double r = (P.rewards == BB_REWARD_ADDITIONS) ? -(double)a : -1.0;
        const double d = acc.disc;
        acc.ret = __dadd_rn(acc.ret, __dmul_rn(d, r)); acc.disc = __dmul_rn(d, A.gamma);
        if (trace && steps < A.trace_cap) trace[steps] = make_int4(pi, pj, a, e.nP);
      }
      steps++; adds += a;
    }
    __syncthreads();
    if (tid < 32) {   // warp 0: episode record, checksums, reduced Groebner basis (the warp routines of bb_device.cuh)
      const int nonzero = e.nG - g_start, zero = steps - nonzero;
      env_store(P, slot, e);
      __syncwarp();
      const GHeadMem* gh = ENV_PTR(GHeadMem, e, P, o_ghead);
      const unsigned long long bh = warp_terms_hash<NV>(ENV_PTR(uint64_t, e, P, o_tkey), ENV_PTR(uint32_t, e, P, o_tcoef),
                                                        e.nT, reinterpret_cast<const int*>(&gh[0].len),
                                                        (int)(sizeof(GHeadMem) / sizeof(int)), e.nG);
      unsigned long long gbh = 0; int gp = 0, gt = 0;
      int status = e.status;
      if (A.compute_gb && status == BB_STATUS_DONE) {
        if (warp_final_gb<NV>(P, slot, row)) {
          gp = P.gcount[2 * slot]; gt = P.gcount[2 * slot + 1];
          gbh = warp_terms_hash<NV>(P.gkey + (size_t)slot * P.max_terms, P.gcoef + (size_t)slot * P.max_terms, gt,
                                    P.glen + (size_t)slot * P.max_basis, 1, gp);
        } else {
          status = BB_STATUS_OVERFLOW_SCRATCH;
        }
      }
      if (A.gb_sink.lens_dev || A.basis_sink.lens_dev) warp_export_episode<NV>(P, A, slot, ep, status);
      if (tid == 0) {
        const unsigned long long th = acc.th; const double ret = acc.ret;
        bb_episode_stats o;
        o.steps = steps; o.additions = adds; o.zero_reductions = zero; o.nonzero_reductions = nonzero;
        o.nbasis = e.nG; o.nterms = e.nT; o.status = status; o.rerolls = S.st[b].rerolls;
        o.trace_hash = th; o.basis_hash = bh; o.gb_hash = gbh; o.gb_polys = gp; o.gb_terms = gt;
        o.discounted_return = ret;
        A.out[ep] = o;
        BBEnvState& St = P.st[slot];
        St.status = status; St.steps = steps; St.adds = adds; St.zero = zero; St.nonzero = nonzero; St.trace_hash = th;
        St.disc_return = ret; St.rerolls = o.rerolls;
        row[CT_STEPS] += (unsigned)steps; row[CT_ADDS] += (unsigned)adds; row[CT_NONZERO] += (unsigned)nonzero;
        row[CT_ZERO] += (unsigned)zero; row[CT_EPISODES] += 1;
      }
      ct.spill(row);
    } else {
      ct.clear();
    }
    __syncthreads();
  }
#ifdef BBW_INSTR
  if (tid == 0) printf("rounds %lld, with table entries %lld (sum of the table lengths %lld), consolidations %lld (their rounds %lld), streams opened in the table %lld\n", ws.n_rounds, ws.n_trounds, ws.sum_T, ws.n_consol, ws.n_crounds, ws.n_topen);
#endif
#ifdef BBW_CLOCK
  if ((tid & 31) == 0) printf("warp %d: before the barrier %lld, barrier + fold %lld, post-processing %lld, outside the rounds %lld cycles; steps: select %lld, pair removal %lld, reduction %lld, update %lld\n", tid >> 5, ws.cw, ws.cb, ws.cp, ws.co, ws.s_sel, ws.s_take, ws.s_red, ws.s_upd);
#endif
  __syncthreads();
  if (tid < CT_COUNT && sh[0][tid]) atomicAdd(&P.counters[tid], sh[0][tid]);
}

// max of doubles through a CAS loop (order independent, hence deterministic)
__device__ __forceinline__ void atomic_max_double(double* addr, double v) {
  unsigned long long* a = reinterpret_cast<unsigned long long*>(addr);
  unsigned long long old = *a;
  while (__longlong_as_double((long long)old) < v) {
    const unsigned long long seen = atomicCAS(a, old, (unsigned long long)__double_as_longlong(v));
    if (seen == old) break;
    old = seen;
  }
}

// BuchbergerEnv::value (buchberger.cpp:332-351): the discounted return of finishing each environment's episode from
// its CURRENT state under a built-in strategy.  Tasks (env, rollout) are pulled from a queue by persistent worker
// warps; a worker forks the environment into its own arena F (the live environments are not modified), runs the
// loop of buchberger() (:243-263) and folds the return into value[env] with max ("sample": :333-341).
template <int NV>
__global__ void __launch_bounds__(BB_THREADS, BB_MIN_BLOCKS) k_value(const __grid_constant__ BBParams P,
                                                                    const __grid_constant__ BBParams F,
                                                                    const __grid_constant__ BBValueArgs A) {
  __shared__ unsigned long long sh[BB_WARPS][CT_COUNT];
  __shared__ BBEpisodeAcc acc_sh[BB_WARPS];
  hot_init(F);
  unsigned long long* row = counters_row(sh);
  BBEpisodeAcc& acc = acc_sh[threadIdx.x >> 5];
  const int w = (blockIdx.x * BB_THREADS + threadIdx.x) >> 5;
  const int lane = bb_lane();
  if (w < F.num_envs) {
    Ctr ct; ct.clear();
    for (;;) {
      int t = 0;
      if (lane == 0) t = atomicAdd(A.queue, 1);
      t = __shfl_sync(BB_FULL, t, 0);
      if (t >= A.ntasks) break;
      const int env = t / A.rollouts, r = t - env * A.rollouts;
      Env e; env_load(P, env, e);
      double ret = 0.0;
      if (e.status == BB_STATUS_RUNNING) {
        unsigned char* db = F.arena + (size_t)w * F.slot_stride;
        warp_copy_env(F, db, P, e.base, e);
        e.base = db;
        __syncwarp();
        int strategy = A.strategy, seed = A.sel_seed_base + r;
        if (strategy == BB_VALUE_SAMPLE) { strategy = r == 0 ? BB_SELECT_DEGREE : BB_SELECT_RANDOM; seed = A.sel_seed_base + r - 1; }
        if (lane == 0) { acc.th = 0ull; acc.ret = 0.0; acc.disc = 1.0; acc.sel_rng = rng_seed(seed); }
        __syncwarp();
        int steps = 0, adds = 0;
        run_episode<NV>(F, e, strategy, A.max_steps, A.gamma, acc, ct, steps, adds, nullptr, 0);
        __syncwarp();
        ret = acc.ret;
        if (e.status != BB_STATUS_DONE && !(A.max_steps && steps >= A.max_steps)) ret = __longlong_as_double(0x7ff8000000000000LL);  // fault: NaN
      }
      if (lane == 0) {
        if (ret != ret) A.value[env] = ret;  // NaN marks an overflowed rollout (never silently wrong)
        else atomic_max_double(&A.value[env], ret);
      }
      ct.clear();  // rollouts of value() are not part of the environments' traffic counters
      __syncwarp();
    }
  }
  (void)row;
}

// The policy head on the current state of every environment (see bb_policy.cuh).
template <int NV, int UPL>
__global__ void __launch_bounds__(BB_THREADS) k_policy(const __grid_constant__ BBParams P, const __grid_constant__ BBPolicy W,
                                                       unsigned long long counter, int32_t* __restrict__ actions,
                                                       float* __restrict__ logp, float* __restrict__ logits, int pmax) {
  extern __shared__ float wsm[];
  policy_load_weights(W, P.cols, wsm);
  const int slot = (blockIdx.x * BB_THREADS + threadIdx.x) >> 5;
  if (slot >= P.num_envs) return;
  Env e; env_load(P, slot, e);
  int a = 0; float lp = 0.0f;
  if (e.status == BB_STATUS_RUNNING)
    a = warp_policy<NV, UPL>(P, e, wsm, W.greedy, policy_uniform(W.seed, (unsigned long long)slot, counter), lp,
                             logits ? logits + (size_t)slot * pmax : nullptr, pmax);
  if (bb_lane() == 0) { actions[slot] = a; if (logp) logp[slot] = lp; }
}

// Fused rollout (the loop of pg.Agent.run_episode, pg.py:451-472, for every environment at once): each warp runs T
// steps of its environment -- policy head, categorical sample, step, auto-reset -- with no host round trip and no
// synchronisation between environments.  Trajectories are written environment-major.
template <int NV, int UPL>
__global__ void __launch_bounds__(BB_THREADS, BB_ROLLOUT_MIN_BLOCKS) k_rollout(const __grid_constant__ BBParams P,
                                                           const __grid_constant__ BBRolloutArgs A) {
  extern __shared__ float wsm[];
  __shared__ unsigned long long sh[BB_WARPS][CT_COUNT];
  hot_init(P);
  policy_load_weights(A.W, P.cols, wsm);
  unsigned long long* row = counters_row(sh);
  const int slot = (blockIdx.x * BB_THREADS + threadIdx.x) >> 5;
  const int lane = bb_lane();
  if (slot < P.num_envs) {
    Env e; env_load(P, slot, e);
    Ctr ct; ct.clear();
    if (e.status != BB_STATUS_RUNNING && P.auto_reset) {  // a slot that was never reset (or finished before the call)
      warp_next_episode<NV>(P, slot, row);
      env_load(P, slot, e);
    }
#pragma unroll 1
    for (int t = 0; t < A.T; t++) {
      const size_t o = (size_t)slot * A.T + t;
      if (A.lengths && lane == 0) A.lengths[o] = e.nP;
      if (A.obs) warp_observe<NV>(P, e, A.obs + o * A.pmax * P.cols, A.pmax, ct);
      int a = -1; float lp = 0.0f; double r = 0.0;
      if (e.status == BB_STATUS_RUNNING) {
        a = warp_policy<NV, UPL>(P, e, wsm, A.W.greedy, policy_uniform(A.W.seed, (unsigned long long)slot, A.counter0 + t),
                                 lp, nullptr, 0);
        r = step_and_account<NV>(P, slot, e, a, ct, row);
      }
      const bool fin = e.status != BB_STATUS_RUNNING;
      if (lane == 0) {
        if (A.actions) A.actions[o] = a;
        if (A.logp) A.logp[o] = lp;
        if (A.reward) A.reward[o] = (float)r;
        if (A.done) A.done[o] = fin ? 1 : 0;
      }
      if (fin && P.auto_reset) {  // same convention as k_step: the next state is the first state of the next episode
        env_store(P, slot, e);
        __syncwarp();
        warp_next_episode<NV>(P, slot, row);
        env_load(P, slot, e);
      }
    }
    env_store(P, slot, e);
    ct.spill(row);
  }
  counters_flush(P, sh);
}

// ------------------------------------------------------------------------------------------------ reduce(g, F)
// Packs n int32 terms (exponent rows of NV, coefficients) into (k, c), lane-strided.  Returns 0, -1 (a coefficient outside
// [1, p) or a negative exponent) or BB_STATUS_OVERFLOW_EXPONENT (an exponent above emax or a degree above dmax).
template <int NV>
__device__ __forceinline__ int reduce_pack_terms(const BBField& F, const int32_t* __restrict__ ex, const int32_t* __restrict__ cf,
                                                 long long n, uint64_t* __restrict__ k, uint32_t* __restrict__ c) {
  typedef KL<NV> K;
  bool bad = false, ovf = false;
#pragma unroll 1
  for (long long t = bb_lane(); t < n; t += 32) {
    const int32_t co = cf[t];
    bad |= co <= 0 || (uint32_t)co >= F.p;
    uint64_t key = 0ull; uint32_t deg = 0u;
#pragma unroll
    for (int v = 0; v < NV; v++) {
      const int32_t x = ex[t * NV + v];
      bad |= x < 0;
      ovf |= x > (int32_t)K::emax;
      key |= (uint64_t)((uint32_t)x & K::fmask) << (K::eshift + v * K::w);
      deg += (uint32_t)x & K::fmask;
    }
    ovf |= deg > K::dmax;
    k[t] = key | ((uint64_t)(K::dmax - (deg & K::dmax)) << K::dshift);
    c[t] = (uint32_t)co;
  }
  if (__any_sync(BB_FULL, bad)) return -1;
  return __any_sync(BB_FULL, ovf) ? BB_STATUS_OVERFLOW_EXPONENT : 0;
}

// Stages divisor list w into the worker's slot: terms at the start of the term arena, one head record per polynomial
// (1/LC, second term, offset, length; sugar 0), and the reducer list rlm / ridx in scan order -- as given, or stable
// ascending by lead monomial when A.sorted (the order of G_ under sort_reducers, buchberger.cpp:308-311).  Returns 0 and
// the list's polynomial and term counts, or the status every query of the list gets.
template <int NV>
__device__ __forceinline__ int reduce_stage_list(const BBParams& P, const BBReduceArgs& A, const Env& e, int w, int& nF, int& nT) {
  const int lane = bb_lane();
  const long long p0 = A.list_off[w], p1 = A.list_off[w + 1];
  nF = 0; nT = 0;
  if (p0 < 0 || p1 < p0) return -1;
  if (p1 - p0 > P.max_basis) return BB_STATUS_OVERFLOW_BASIS;
  const long long t0 = A.poly_off[p0], t1 = A.poly_off[p1];
  if (t0 < 0 || t1 < t0) return -1;
  if (t1 - t0 > P.max_terms) return BB_STATUS_OVERFLOW_TERMS;
  uint64_t* tk = ENV_PTR(uint64_t, e, P, o_tkey);
  uint32_t* tc = ENV_PTR(uint32_t, e, P, o_tcoef);
  const int rc = reduce_pack_terms<NV>(P.F, A.exps + t0 * NV, A.coefs + t0, t1 - t0, tk, tc);
  if (rc) return rc;
  __syncwarp();
  const int m = (int)(p1 - p0);
  GHeadMem* gh = ENV_PTR(GHeadMem, e, P, o_ghead);
  bool bad = false;
#pragma unroll 1
  for (int i = lane; i < m; i += 32) {   // every polynomial non-zero, inside the list's terms, strictly descending
    const long long a = A.poly_off[p0 + i] - t0, b = A.poly_off[p0 + i + 1] - t0;
    if (a < 0 || b <= a || b > t1 - t0) { bad = true; continue; }
    for (long long t = a; t + 1 < b; t++) bad |= tk[t] >= tk[t + 1];
    const uint64_t lm = tk[a], k1 = b - a > 1 ? tk[a + 1] : 0ull;
    const uint32_t c1 = b - a > 1 ? tc[a + 1] : 0u;
    reinterpret_cast<uint4*>(gh + i)[0] = make_uint4((uint32_t)lm, (uint32_t)(lm >> 32), (uint32_t)k1, (uint32_t)(k1 >> 32));
    reinterpret_cast<uint4*>(gh + i)[1] = make_uint4((uint32_t)bb_global(P.invtab)[tc[a]] | (c1 << 16), 0u, (uint32_t)a,
                                                     (uint32_t)(b - a));
  }
  if (__any_sync(BB_FULL, bad)) return -1;
  __syncwarp();
  uint64_t* rlm = ENV_PTR(uint64_t, e, P, o_rlm);
  uint32_t* ridx = ENV_PTR(uint32_t, e, P, o_ridx);
#pragma unroll 1
  for (int i = lane; i < m; i += 32) {
    const uint64_t li = gh[i].lm;
    int pos = i;
    if (A.sorted) {   // ascending lead monomial == descending key; equal lead monomials keep their order
      pos = 0;
      for (int j = 0; j < m; j++) { const uint64_t lj = gh[j].lm; pos += lj > li || (lj == li && j < i); }
    }
    rlm[pos] = li; ridx[pos] = (uint32_t)i;
  }
  __syncwarp();
  nF = m; nT = (int)(t1 - t0);
  return 0;
}

// reduce(g, F) (buchberger.cpp:24-49) of query q by the list staged in the slot (nF polynomials on nT terms): the dividend goes
// to scratch half 0, warp_reduce runs on it, the remainder lands behind the list's terms.  Returns the query's status.
template <int NV>
__device__ __forceinline__ int reduce_query(const BBParams& P, const BBReduceArgs& A, Env& e, int q, int nF, int nT, int& steps,
                                            int& rlen, Ctr& ct) {
  typedef KL<NV> K;
  steps = 0; rlen = 0;
  const long long a0 = A.q_off[q], a1 = A.q_off[q + 1];
  if (a0 < 0 || a1 < a0) return -1;
  if (a1 - a0 > P.max_poly_terms) return BB_STATUS_OVERFLOW_SCRATCH;
  const int n = (int)(a1 - a0);
  uint64_t* hk = ENV_PTR(uint64_t, e, P, o_hkey);
  uint32_t* hc = ENV_PTR(uint32_t, e, P, o_hcoef);
  const int rc = reduce_pack_terms<NV>(P.F, A.q_exps + a0 * NV, A.q_coefs + a0, n, hk, hc);
  if (rc) return rc;
  __syncwarp();
  bool bad = false;
#pragma unroll 1
  for (int t = bb_lane(); t + 1 < n; t += 32) bad |= hk[t] >= hk[t + 1];
  if (__any_sync(BB_FULL, bad)) return -1;
  Dividend h;
  h.k0 = h.k1 = 0; h.c0 = h.c1 = 0; h.sug = 0;
  dividend_from_scratch(P, e, h, n, 0);
  e.guard = 0;
  rlen = warp_reduce<NV>(P, e, h, ENV_PTR(uint64_t, e, P, o_rlm), ENV_PTR(uint32_t, e, P, o_ridx), nF, A.sorted != 0,
                         ENV_PTR(uint64_t, e, P, o_tkey) + nT, ENV_PTR(uint32_t, e, P, o_tcoef) + nT, P.max_terms - nT, steps, ct);
  if (rlen < 0 || (e.guard & K::g_all))
    return rlen == -1 ? BB_STATUS_OVERFLOW_SCRATCH : (rlen == -2 ? BB_STATUS_OVERFLOW_TERMS : BB_STATUS_OVERFLOW_EXPONENT);
  return BB_STATUS_DONE;
}

// bb_reduce: persistent worker warps, one slot each.  Per query: steps, remainder length and status (nothing else is written
// for a query that does not end BB_STATUS_DONE), the remainder to the sink as entry q.  The traffic counters and `additions`
// count the queries that end done; env_steps and episodes are not touched.
template <int NV>
__global__ void __launch_bounds__(BB_THREADS, BB_MIN_BLOCKS) k_reduce(const __grid_constant__ BBParams P,
                                                                     const __grid_constant__ BBReduceArgs A) {
  __shared__ unsigned long long sh[BB_WARPS][CT_COUNT];
  unsigned long long* row = counters_row(sh);
  const int slot = (blockIdx.x * BB_THREADS + threadIdx.x) >> 5;
  const int lane = bb_lane();
  if (slot < P.num_envs) {
    Env e;
    e.base = bb_global(P.arena + (size_t)slot * P.slot_stride);
    e.nG = e.nP = e.nT = 0; e.status = BB_STATUS_RUNNING; e.guard = 0;
    Ctr ct; ct.clear();
    int staged = -1, lstat = 0, nF = 0, nT = 0;
    for (;;) {
      int q0 = 0;
      if (lane == 0) q0 = atomicAdd(A.queue, A.chunk);
      q0 = __shfl_sync(BB_FULL, q0, 0);
      if (q0 >= A.nq) break;
      const int q1 = q0 + A.chunk < A.nq ? q0 + A.chunk : A.nq;
#pragma unroll 1
      for (int q = q0; q < q1; q++) {
        const int w = A.which[q];
        int status = -1, steps = 0, rlen = 0;
        if ((unsigned)w < (unsigned)A.nlists) {
          if (w != staged) { lstat = reduce_stage_list<NV>(P, A, e, w, nF, nT); staged = w; }
          status = lstat ? lstat : reduce_query<NV>(P, A, e, q, nF, nT, steps, rlen, ct);
        }
        const bool done = status == BB_STATUS_DONE;
        if (lane == 0) {
          A.steps[q] = done ? steps : 0; A.rlen[q] = done ? rlen : 0; A.status[q] = status;
          if (done) row[CT_ADDS] += (unsigned)steps;
        }
        if (done) {
          ct.spill(row);
          __syncwarp();
          if (A.sink.lens_dev)
            warp_export_polys<NV>(ENV_PTR(uint64_t, e, P, o_tkey) + nT, ENV_PTR(uint32_t, e, P, o_tcoef) + nT, A.rlen + q, 1, 1,
                                  rlen, A.sink, q);
        } else {
          ct.clear();
        }
        __syncwarp();
      }
    }
  }
  counters_flush(P, sh);
}

// ------------------------------------------------------------------------------------------------ launchers
static inline int grid_for_warps(int nwarps) { return (nwarps + BB_WARPS - 1) / BB_WARPS; }

template <int NV>
struct BBLaunch {
  static cudaError_t reset(const BBParams& P, const uint8_t* mask, int nwarps, cudaStream_t s) {
    k_reset<NV><<<grid_for_warps(nwarps), BB_THREADS, 0, s>>>(P, mask);
    return cudaGetLastError();
  }
  static cudaError_t step(const BBParams& P, const int* actions, double* reward, uint8_t* done, const int* active, int nwarps,
                          cudaStream_t s) {
    k_step<NV><<<grid_for_warps(nwarps), BB_THREADS, 0, s>>>(P, actions, reward, done, active);
    return cudaGetLastError();
  }
  static cudaError_t step_obs(const BBParams& P, const int* actions, int action0, double* reward, uint8_t* done, int32_t* obs,
                              int32_t* lengths, int pmax, int pad, int do_step, const int* active, unsigned* ready,
                              unsigned ticket, int nwarps, cudaStream_t s) {
    k_step_obs<NV><<<grid_for_warps(nwarps), BB_THREADS, 0, s>>>(P, actions, action0, reward, done, obs, lengths, pmax, pad, do_step,
                                                                active, ready, ticket);
    return cudaGetLastError();
  }
  static cudaError_t serve(const BBParams& P, BBMailbox* mb, unsigned long long idle_ns, cudaStream_t s) {
    k_serve<NV><<<1, 32, 0, s>>>(P, mb, idle_ns);
    return cudaGetLastError();
  }
  static cudaError_t prefill(const BBParams& P, const BBParams& S, int period, cudaStream_t s) {
    k_prefill<NV><<<(P.num_envs + BB_PREP_THREADS - 1) / BB_PREP_THREADS, BB_PREP_THREADS, 0, s>>>(P, S, period);
    return cudaGetLastError();
  }
  static cudaError_t select(const BBParams& P, int strategy, int* actions, int nwarps, cudaStream_t s) {
    k_select<NV><<<grid_for_warps(nwarps), BB_THREADS, 0, s>>>(P, strategy, actions);
    return cudaGetLastError();
  }
  static cudaError_t observe(const BBParams& P, int32_t* obs, int32_t* lengths, int pmax, int nwarps, cudaStream_t s) {
    k_observe<NV><<<grid_for_warps(nwarps), BB_THREADS, 0, s>>>(P, obs, lengths, pmax);
    return cudaGetLastError();
  }
  static cudaError_t final_gb(const BBParams& P, int slot, int* ok_out, cudaStream_t s) {
    k_final_gb<NV><<<1, 32, 0, s>>>(P, slot, ok_out);
    return cudaGetLastError();
  }
  // The runner of batch i and the preparation of batch i + 1 are meant to share the SMs (bb_prepare on a side stream).  An SM
  // runs CTAs of two kernels side by side only when both ask for the same shared-memory / L1 split, and by default the
  // driver picks the split per kernel from its own shared-memory use (measured, profiles/README.md r2: the preparation sat
  // in the queue until the runner's CTAs left).  Every kernel of the pipeline therefore states the same preference.
  static void same_carveout() {
    static bool done = false;
    if (done) return;
    done = true;
    // -> the 16 KB split: three general runner CTAs use ~6.5 KB of it (run_worker's arrays and the 1 KB reserved per CTA)
    const int pct = 7;
    static_assert(BB_TWO_MIN_BLOCKS * (BB_TWO_WARPS * (CT_COUNT * 8 + sizeof(BBEpisodeAcc)) + 1024) <= 16 * 1024,
                  "the 16 KB split holds BB_TWO_MIN_BLOCKS two-term runner CTAs");
    cudaFuncSetAttribute(k_run<NV>, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
    cudaFuncSetAttribute(k_run<NV, true>, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
    cudaFuncSetAttribute(k_run<NV, false, true>, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
    cudaFuncSetAttribute(k_run<NV, true, true>, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
    cudaFuncSetAttribute(k_prepare<NV>, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
    cudaFuncSetAttribute(k_prepare_lanes<NV>, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
    cudaFuncSetAttribute(k_order<NV>, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
    cudaFuncSetAttribute(k_reduce<NV>, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
  }
  static cudaError_t prepare(const BBParams& S, const BBRunArgs& A, cudaStream_t s) {
    same_carveout();
    // binomial distributions with few generators: one thread per episode; everything else: one warp per episode
    if (S.dist.enabled && S.dist.kind == 0 && S.dist.s <= BB_PREP_S && !A.prepare_by_warp)
      k_prepare_lanes<NV><<<(A.episodes + BB_PREP_THREADS - 1) / BB_PREP_THREADS, BB_PREP_THREADS, 0, s>>>(S, A);
    else
      k_prepare<NV><<<grid_for_warps(A.episodes), BB_THREADS, 0, s>>>(S, A);
    k_order<NV><<<std::min(64, (A.episodes + 1023) / 1024), BB_LPT_BUCKETS, 0, s>>>(A);
    return cudaGetLastError();
  }
  static cudaError_t run(const BBParams& P, const BBParams& S, const BBRunArgs& A, int nwarps, cudaStream_t s) {
    same_carveout();
    const bool ex = A.gb_sink.lens_dev || A.basis_sink.lens_dev;
    if (A.two_term) {
      const int g = (nwarps + BB_TWO_WARPS - 1) / BB_TWO_WARPS;
      if (ex) k_run<NV, true, true><<<g, BB_TWO_WARPS * 32, 0, s>>>(P, S, A);
      else k_run<NV, false, true><<<g, BB_TWO_WARPS * 32, 0, s>>>(P, S, A);
    } else {
      if (ex) k_run<NV, true><<<grid_for_warps(nwarps), BB_THREADS, 0, s>>>(P, S, A);
      else k_run<NV><<<grid_for_warps(nwarps), BB_THREADS, 0, s>>>(P, S, A);
    }
    return cudaGetLastError();
  }
  static int wide_ctas_per_sm() {
    const size_t sm = sizeof(WideStreams);
    if (cudaFuncSetAttribute(k_run_wide<NV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm) != cudaSuccess) return 0;
    int blocks = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, k_run_wide<NV>, BBW_THREADS, sm) != cudaSuccess) return 0;
    return blocks;
  }
  static cudaError_t run_wide(const BBParams& P, const BBParams& S, const BBRunArgs& A, int nctas, cudaStream_t s) {
    const size_t sm = sizeof(WideStreams);
    cudaError_t e = cudaFuncSetAttribute(k_run_wide<NV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    if (e != cudaSuccess) return e;
    k_run_wide<NV><<<nctas, BBW_THREADS, sm, s>>>(P, S, A);
    return cudaGetLastError();
  }
  static cudaError_t value(const BBParams& P, const BBParams& F, const BBValueArgs& A, int nwarps, cudaStream_t s) {
    k_value<NV><<<grid_for_warps(nwarps), BB_THREADS, 0, s>>>(P, F, A);
    return cudaGetLastError();
  }
  static size_t policy_smem(const BBParams& P, int hidden) { return sizeof(float) * (size_t)policy_smem_floats(P.cols, hidden); }
  // The policy kernels exist for hidden = 32 * UPL, UPL in {1, 2, 4, 8}: body(std::integral_constant<int, UPL>()) for the UPL
  // of `hidden`, `bad` for any other width.
  template <class R, class Body>
  static R with_upl(int hidden, R bad, Body body) {
    switch (hidden >> 5) {
      case 1: return body(std::integral_constant<int, 1>());
      case 2: return body(std::integral_constant<int, 2>());
      case 4: return body(std::integral_constant<int, 4>());
      case 8: return body(std::integral_constant<int, 8>());
    }
    return bad;
  }
  static cudaError_t policy(const BBParams& P, const BBPolicy& W, unsigned long long counter, int32_t* actions, float* logp,
                            float* logits, int pmax, int nwarps, cudaStream_t s) {
    const size_t sm = policy_smem(P, W.hidden);
    return with_upl(W.hidden, cudaErrorInvalidValue, [&](auto upl) {
      constexpr int UPL = decltype(upl)::value;
      if (sm > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(k_policy<NV, UPL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
        if (e != cudaSuccess) return e;
      }
      k_policy<NV, UPL><<<grid_for_warps(nwarps), BB_THREADS, sm, s>>>(P, W, counter, actions, logp, logits, pmax);
      return cudaGetLastError();
    });
  }
  static cudaError_t rollout(const BBParams& P, const BBRolloutArgs& A, int nwarps, cudaStream_t s) {
    const size_t sm = policy_smem(P, A.W.hidden);
    return with_upl(A.W.hidden, cudaErrorInvalidValue, [&](auto upl) {
      constexpr int UPL = decltype(upl)::value;
      if (sm > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(k_rollout<NV, UPL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
        if (e != cudaSuccess) return e;
      }
      k_rollout<NV, UPL><<<grid_for_warps(nwarps), BB_THREADS, sm, s>>>(P, A);
      return cudaGetLastError();
    });
  }
  // resident warps per SM of the general (two == 0) or the two-term k_run (the instantiations with sinks have the same bounds)
  static int run_warps_per_sm(int two) {
    same_carveout();
    int blocks = 0;
    const cudaError_t e = two ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, k_run<NV, false, true>, BB_TWO_WARPS * 32, 0)
                              : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, k_run<NV>, BB_THREADS, 0);
    if (e != cudaSuccess) return -1;
    return blocks * (two ? BB_TWO_WARPS : BB_WARPS);
  }
  static cudaError_t reduce(const BBParams& P, const BBReduceArgs& A, int nwarps, cudaStream_t s) {
    same_carveout();
    k_reduce<NV><<<grid_for_warps(nwarps), BB_THREADS, 0, s>>>(P, A);
    return cudaGetLastError();
  }
  static cudaError_t run_policy(const BBParams& P, const BBParams& S, const BBRunArgs& A, const BBPolicy& W,
                                unsigned long long counter0, int nwarps, cudaStream_t s) {
    const size_t sm = policy_smem(P, W.hidden);
    return with_upl(W.hidden, cudaErrorInvalidValue, [&](auto upl) {
      constexpr int UPL = decltype(upl)::value;
      if (sm > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(k_run_policy<NV, UPL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
        if (e != cudaSuccess) return e;
      }
      k_run_policy<NV, UPL><<<grid_for_warps(nwarps), BB_THREADS, sm, s>>>(P, S, A, W, counter0);
      return cudaGetLastError();
    });
  }
  static int run_policy_warps_per_sm(const BBParams& P, int hidden) {
    const size_t sm = policy_smem(P, hidden);
    return with_upl(hidden, -1, [&](auto upl) {
      constexpr int UPL = decltype(upl)::value;
      if (sm > 48 * 1024 &&
          cudaFuncSetAttribute(k_run_policy<NV, UPL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm) != cudaSuccess)
        return -1;
      int blocks = 0;
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, k_run_policy<NV, UPL>, BB_THREADS, sm) != cudaSuccess) return -1;
      return blocks * BB_WARPS;
    });
  }
  static const BBKernelTable* table() {
    static const BBKernelTable t = {NV, KL<NV>::w, KL<NV>::dw, KL<NV>::dshift, KL<NV>::eshift,
                                    &reset, &step, &step_obs, &serve, &prefill, &select, &observe, &final_gb, &prepare, &run, &run_wide, &wide_ctas_per_sm, &value, &policy,
                                    &rollout,
                                    &run_warps_per_sm, &reduce, &run_policy, &run_policy_warps_per_sm};
    return &t;
  }
};
#endif  // BB_NV
