/*
 * bbenv.h -- C-ABI of libbbenv.so, the B200-native (sm_100a) batched Buchberger environment.
 *
 * This is the drop-in boundary for the reference's native environment, i.e. what the reference's
 * Cython binding (deepgroebner/buchberger.pxd:8-18, deepgroebner/wrapped.pyx:11-38) binds today:
 *
 *   reference (one episode, host)                           this library (N episodes, device)
 *   ------------------------------------------------------  -----------------------------------------
 *   LeadMonomialsEnv(string,bint,bint,int) pxd:11           bb_create(cfg)  (+ bb_set_distribution)
 *   ~LeadMonomialsEnv                                       bb_destroy
 *   void seed(int)                       pxd:15             bb_seed / bb_seed_on
 *   void reset()                         pxd:13             bb_reset / bb_set_ideals
 *   double step(int)                     pxd:14             bb_step
 *   vector[int] state, int cols          pxd:17-18          bb_observe, bb_cols
 *   double value(string,double)          pxd:16             bb_value (fork + rollouts from the live state);
 *                                                             bb_rollout_value (every state of a fused rollout)
 *   LeadMonomialsEnv(const&)  (copy())   pxd:12             bb_copy_env
 *   buchberger(F, selection, ...)  buchberger.h:127-147     bb_run_export (whole episodes, all nine SelectionTypes;
 *                                                             every episode's reduced basis into a device sink), bb_run
 *   policy_model(state) + categorical   pg.py:323-326       bb_policy_pmlp / bb_rollout (PMLP head, networks.py:522-571)
 *   TrajectoryBuffer states (unpadded)  pg.py:162-241       bb_rollout_rows (every state at its own row count)
 *   pg.Agent.run_episode to completion  pg.py:451-472       bb_run_policy (whole episodes, the PMLP head selecting, with
 *                                                             bb_run_export's records, traces and sinks)
 *   BuchbergerEnv::G, ::P   buchberger.h:195-196            bb_download_basis, bb_pairs
 *   buchberger(...) -> interreduce(minimalize(G))           bb_final_gb
 *       buchberger.cpp:265
 *   reduce(g, F) -> (r, ReduceStats)   buchberger.h:26-28   bb_reduce (batches of dividends against device-resident lists)
 *
 * Conventions: plain pointers and sizes only (no torch types).  Every entry point returns 0 on success and a
 * negative code otherwise; bb_last_error() gives the message.  Pointers named *_dev are DEVICE pointers in the
 * handle's device; all others are HOST pointers.  Work is enqueued on `stream` (a cudaStream_t passed as
 * void*; NULL = the legacy default stream); calls taking host output pointers synchronise that stream.
 * A handle is single-owner and not thread-safe (the reference env has no threading either).  Per-environment
 * faults (bad action, arena / exponent overflow) never abort: they set that environment's status word
 * (BB_STATUS_*), the environment stops stepping and reports done.
 */
#ifndef BBENV_H
#define BBENV_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BB_ABI_VERSION 3

/* EliminationType, buchberger.h:58 */
enum { BB_ELIM_GEBAUERMOELLER = 0, BB_ELIM_LCM = 1, BB_ELIM_NONE = 2 };
/* RewardType, buchberger.h:93 */
enum { BB_REWARD_ADDITIONS = 0, BB_REWARD_REDUCTIONS = 1 };
/* SelectionType, buchberger.h:111 (same order).  BB_SELECT_RANDOM draws choice() (ideals.h:68-73) from a
 * per-episode minstd_rand0 stream, i.e. buchberger(..., seed) of buchberger.cpp:190-197. */
enum { BB_SELECT_FIRST = 0, BB_SELECT_DEGREE = 1, BB_SELECT_NORMAL = 2, BB_SELECT_SUGAR = 3, BB_SELECT_RANDOM = 4,
       BB_SELECT_LAST = 5, BB_SELECT_CODEGREE = 6, BB_SELECT_STRANGE = 7, BB_SELECT_SPICE = 8,
       BB_VALUE_SAMPLE = 100 /* bb_value only: value("sample"), buchberger.cpp:333-341 */ };
/* DistributionType, ideals.h:40 */
enum { BB_DIST_UNIFORM = 0, BB_DIST_WEIGHTED = 1, BB_DIST_MAXIMUM = 2 };

/* per-environment status word */
enum {
  BB_STATUS_EMPTY = 0,     /* slot holds no episode */
  BB_STATUS_RUNNING = 1,   /* pair set non-empty */
  BB_STATUS_DONE = 2,      /* pair set empty: episode finished */
  BB_STATUS_BAD_ACTION = 3,/* action index outside [0, |P|)  (UB in the reference, buchberger.cpp:399) */
  BB_STATUS_OVERFLOW_BASIS = 4,
  BB_STATUS_OVERFLOW_PAIRS = 5,
  BB_STATUS_OVERFLOW_TERMS = 6,
  BB_STATUS_OVERFLOW_EXPONENT = 7, /* a packed exponent/degree field would wrap: never silently wrong */
  BB_STATUS_OVERFLOW_SCRATCH = 8,
  BB_STATUS_TRUNCATED = 9   /* cut by bb_set_max_episode_length (pg.py:470-471): done, not finished */
};
#define BB_STATUS_COUNT 10

typedef struct bb_config {
  int abi_version;    /* BB_ABI_VERSION */
  int device;         /* CUDA device ordinal */
  int nvars;          /* n, 1..8 (polynomials.h:29 fixes 8 exponent slots) */
  int k;              /* lead monomials shown per polynomial (buchberger.h:224-231); cols = 2*n*k */
  int prime;          /* field characteristic, 2 < p < 65536 (reference: 32003, polynomials.h:10) */
  int elimination;    /* BB_ELIM_* */
  int rewards;        /* BB_REWARD_* */
  int sort_input;     /* buchberger.cpp:301-302 */
  int sort_reducers;  /* buchberger.cpp:308-311, 323-326 */
  int num_envs;       /* N environment slots */
  int max_basis;      /* capacity |G| per env  (<= 65535) */
  int max_pairs;      /* capacity |P| per env */
  int max_terms;      /* capacity of the term arena per env (sum of |g| over G) */
  int max_poly_terms; /* capacity of the dividend scratch (longest intermediate polynomial) */
  int max_gens;       /* capacity of generators per input ideal */
  int max_gen_terms;  /* capacity of terms per input ideal */
} bb_config;

typedef struct bb_handle bb_handle;

/* Work/traffic counters accumulated by the kernels (SURVEY 8(d) algorithmic-bytes model). */
typedef struct bb_counters {
  unsigned long long env_steps;        /* step() transitions executed */
  unsigned long long additions;        /* polynomial additions as the reward counts them (1 per spoly + 1 per reduction) */
  unsigned long long terms_read;       /* |h_in| + |f| (+|g|) over all additions */
  unsigned long long terms_written;    /* |h_out| over all additions */
  unsigned long long lms_scanned;      /* reducer lead monomials examined by divisor searches */
  unsigned long long term_moves;       /* lead terms moved to the remainder */
  unsigned long long update_basis;     /* sum of m over update() calls */
  unsigned long long update_pairs;     /* |P| before + |P_new| over update() calls */
  unsigned long long obs_rows;         /* observation rows written */
  unsigned long long nonzero_reductions;
  unsigned long long zero_reductions;
  unsigned long long episodes;         /* episodes finished */
} bb_counters;

/* Per-episode record written by bb_run / kept per slot (BuchbergerStats, buchberger.h:99-105, plus checksums). */
typedef struct bb_episode_stats {
  int32_t steps;               /* episode length */
  int32_t additions;           /* polynomial_additions  (= -total_reward under Additions) */
  int32_t zero_reductions;
  int32_t nonzero_reductions;
  int32_t nbasis;              /* |G| at the end */
  int32_t nterms;              /* sum of |g| at the end */
  int32_t status;              /* BB_STATUS_* */
  int32_t rerolls;             /* ideals skipped by reset() because P came out empty (buchberger.cpp:313-314) */
  uint64_t trace_hash;         /* checksum of the (i, j, additions) sequence, see "checksums" below */
  uint64_t basis_hash;         /* checksum of the final basis G (all terms, in insertion order) */
  uint64_t gb_hash;            /* checksum of interreduce(minimalize(G)) when bb_run(compute_gb=1), else 0 */
  int32_t gb_polys, gb_terms;  /* its size */
  double discounted_return;    /* sum gamma^t * reward_t (buchberger.cpp:250-251) */
} bb_episode_stats;

int bb_abi_version(void);

/* ---- lifetime */
int bb_create(const bb_config* cfg, bb_handle** out);
void bb_destroy(bb_handle* h);
const char* bb_last_error(const bb_handle* h); /* h may be NULL: last error of bb_create */
int bb_cols(const bb_handle* h);               /* 2*n*k, LeadMonomialsEnv::cols */
int bb_num_envs(const bb_handle* h);
int bb_sm_count(const bb_handle* h);
/* Number of environment slots (warps) of the persistent episode runner that are co-resident on `device`
 * (occupancy of k_run<nvars> x SM count).  Creating the handle with this many slots keeps bb_run to a single wave. */
int bb_resident_envs(int device, int nvars);

/* ---- input ideals
 * bb_set_distribution: the analogue of parse_ideal_dist("n-d-s-{uniform,weighted,maximum}[-consts][-homog][-pure]")
 * (ideals.cpp:103-143) for RandomBinomialIdealGenerator; n must equal cfg.nvars.  Ideals are then drawn ON DEVICE by
 * bb_reset from per-environment minstd_rand0 streams that reproduce libstdc++'s distributions bit-for-bit.
 * bb_seed: stream[e] <- seeds[e] for every environment (BuchbergerEnv::seed, buchberger.h:189); seeds == NULL
 * seeds environment e with base + e. */
int bb_set_distribution(bb_handle* h, int d, int s, int dist, int constants, int homogeneous, int pure);
/* bb_set_distribution_poly: the same for "n-d-s-lam-{uniform,weighted,maximum}[-consts][-homog]", RandomIdealGenerator
 * (ideals.cpp:204-231): s monic polynomials of 2 + Poisson(lam) random terms each, drawn on device with libstdc++'s
 * poisson_distribution stream (mean < 12 branch; lam >= 12 is refused).  cfg.max_gen_terms bounds the terms of one
 * ideal: an ideal that does not fit leaves its environment in BB_STATUS_OVERFLOW_TERMS. */
int bb_set_distribution_poly(bb_handle* h, int d, int s, double lam, int dist, int constants, int homogeneous);
int bb_seed(bb_handle* h, const int32_t* seeds, int base);
/* bb_seed_on: bb_seed (selection == 0) / bb_seed_selection (selection != 0) enqueued on `stream`.  No allocation and no
 * device synchronisation: the reference pattern re-seeds before every episode (randomized_agent.py:141-142).  bb_seed and
 * bb_seed_selection are the same on the legacy default stream. */
int bb_seed_on(bb_handle* h, const int32_t* seeds, int base, int selection, void* stream);
/* bb_seed_selection: the same for the per-environment stream BB_SELECT_RANDOM draws from in bb_select (the `seed`
 * argument of buchberger(), buchberger.cpp:190-197).  Both streams are seeded with base + e at bb_create. */
int bb_seed_selection(bb_handle* h, const int32_t* seeds, int base);

/* bb_set_ideals: explicit ideals, the analogue of FixedIdealGenerator (ideals.h:116-138; buchberger.py:389-394).
 *   count          number of ideals; ideal c goes to environment env_ids[c] (env_ids == NULL: environment c)
 *   ideal_offsets  [count+1]   polynomial index range of each ideal
 *   poly_offsets   [npolys+1]  term index range of each polynomial
 *   exps           [nterms*n]  exponent vectors;  coefs [nterms] in [0,p).  Terms of a polynomial may come in any
 *                  order (they are sorted like the Polynomial ctor, polynomials.cpp:139-145) but must be distinct.
 * The ideals are staged; bb_reset loads them (every reset of that environment replays the same ideal). */
int bb_set_ideals(bb_handle* h, const int32_t* env_ids, int count, const int32_t* ideal_offsets,
                  const int32_t* poly_offsets, const int32_t* exps, const int32_t* coefs);

/* ---- the environment (BuchbergerEnv::reset/step, buchberger.cpp:299-329)
 * bb_reset: mask_dev (uint8[N], NULL = all) selects the environments to reset. */
int bb_reset(bb_handle* h, const uint8_t* mask_dev, void* stream);
/* bb_step: actions_dev int32[N] row indices into each environment's pair list (LeadMonomialsEnv::step(int),
 * buchberger.cpp:398-408).  reward_dev double[N] (-(1+steps) or -1), done_dev uint8[N] (|P| == 0).  Environments
 * that are not RUNNING are skipped (reward 0, done 1). */
int bb_step(bb_handle* h, const int32_t* actions_dev, double* reward_dev, uint8_t* done_dev, void* stream);
/* bb_step_observe: bb_step followed by bb_observe of the new state (after the auto-reset, if enabled) in ONE launch --
 * LeadMonomialsEnv::step(int) as a whole (buchberger.cpp:398-408: step, then the state matrix is rebuilt).  Device
 * buffers as in bb_step / bb_observe (reward_dev, done_dev, obs_dev, lengths_dev may be NULL); rows beyond |P| are -1. */
int bb_step_observe(bb_handle* h, const int32_t* actions_dev, double* reward_dev, uint8_t* done_dev, int32_t* obs_dev,
                    int32_t* lengths_dev, int pmax, void* stream);
/* bb_step_host / bb_reset_host / bb_observe_host: the same calls as the reference's binding makes them -- HOST buffers,
 * synchronous, step + state matrix + done in ONE call (wrapped.pyx:18-26: `step` returns the matrix copied out of
 * LeadMonomialsEnv::state).  One kernel launch and one stream synchronisation per call: the kernel does the step (and the
 * auto-reset, if enabled) and writes the observation of the NEW state; for small batches it reads the actions from and
 * writes the results to pinned host memory in place (N == 1: the action travels in the launch parameters), for large
 * ones there is one async copy each way.  actions_host int32[N]; reward_host double[N], done_host uint8[N],
 * lengths_host int32[N] = |P| after the step, obs_host int32[N, pmax, cols] (any output may be NULL).  pad != 0: rows
 * beyond |P| are -1 (pg.py:217-226); pad == 0: only the first min(|P|, pmax) rows of each environment are written. */
int bb_step_host(bb_handle* h, const int32_t* actions_host, double* reward_host, uint8_t* done_host, int32_t* obs_host,
                 int32_t* lengths_host, int pmax, int pad, void* stream);
int bb_reset_host(bb_handle* h, int32_t* obs_host, int32_t* lengths_host, int pmax, int pad, void* stream);
/* bb_set_serve: a handle of ONE environment answers bb_step_host / bb_reset_host / bb_observe_host through a resident warp
 * (the "environment server") that polls a mailbox in mapped pinned host memory: the host writes the action, the warp runs
 * the step and writes reward, done, |P| and the state matrix back -- a PCIe round trip per call instead of a kernel launch
 * and a synchronisation (the reference's binding is called once per environment step, wrapped.pyx:23-26).  The warp is
 * started on demand (ordered after the work already enqueued on `stream`), leaves after 10 ms without a command, and is
 * joined by every other entry point before it touches the handle.  on = 0: one kernel launch per call.  Default: on when
 * num_envs == 1. */
int bb_set_serve(bb_handle* h, int on);
int bb_observe_host(bb_handle* h, int32_t* obs_host, int32_t* lengths_host, int pmax, int pad, void* stream);
/* bb_select: built-in pair selection (buchberger.cpp:160-241, any BB_SELECT_*): actions_dev int32[N]. */
int bb_select(bb_handle* h, int strategy, int32_t* actions_dev, void* stream);
/* bb_observe: obs_dev int32[N, pmax, cols] padded with -1 (pg.py:217-226), lengths_dev int32[N] = |P|
 * (lead_monomials_vector rows, buchberger.cpp:354-370, 402-406).  Rows beyond pmax are dropped (lengths keeps |P|). */
int bb_observe(bb_handle* h, int32_t* obs_dev, int32_t* lengths_dev, int pmax, void* stream);
/* bb_pairs: pairs_dev int32[N, pmax, 2] = (i, j), padded with -1; lengths_dev int32[N]. */
int bb_pairs(bb_handle* h, int32_t* pairs_dev, int32_t* lengths_dev, int pmax, void* stream);
/* bb_status / bb_stats: status_dev int32[N]; stats_dev bb_episode_stats[N] (running totals of the current episode) */
int bb_status(bb_handle* h, int32_t* status_dev, void* stream);
int bb_stats(bb_handle* h, bb_episode_stats* stats_dev, void* stream);

/* ---- whole episodes on device (the loop of buchberger(), buchberger.cpp:243-263, per environment)
 * bb_run: runs `episodes` episodes to completion with on-device selection.  The handle's N slots act as workers that
 * pull episode e = 0..episodes-1 from a queue (finished slots are refilled at once, so warps stay full); episode e
 * draws its ideal from stream seed = seed_base + e (or seeds_dev[e]) when a distribution is set, or replays staged
 * ideal (e mod staged count; the staged environments must be a prefix 0 .. count-1 of the handle, else the call fails).
 * Calls of more than 65536 episodes go batch by batch, the next batch being prepared on a side stream of the handle
 * while the runner works through the current one.  stats_dev bb_episode_stats[episodes].  trace_dev (optional) int32[trace_episodes,
 * trace_cap, 4] = (i, j, additions, |P| after) for the first trace_episodes episodes, -1 padded.
 * max_steps truncates an episode (0 = unlimited); gamma feeds discounted_return.  With BB_SELECT_RANDOM episode e
 * draws its choices from a minstd_rand0 stream seeded sel_seed_base + e (buchberger(..., seed), buchberger.cpp:190-197). */
int bb_run(bb_handle* h, int strategy, int episodes, int seed_base, const int32_t* seeds_dev, int sel_seed_base,
           int max_steps, double gamma, int compute_gb, bb_episode_stats* stats_dev, int32_t* trace_dev,
           int trace_episodes, int trace_cap, void* stream);

/* A packed, caller-owned device buffer of polynomials (all *_dev pointers in the handle's device). */
typedef struct bb_poly_sink {
  int32_t* lens_dev;            /* [cap_polys]      length of each stored polynomial */
  int32_t* exps_dev;            /* [cap_terms * n]  exponent vectors, int32, n = cfg.nvars */
  int32_t* coefs_dev;           /* [cap_terms]      coefficients in [0, p) */
  int64_t* where_dev;           /* [episodes * 2]   (first polynomial, first term) of episode e of the call, (-1, -1)
                                                    where nothing was stored */
  unsigned long long* used_dev; /* [3] polynomials reserved, terms reserved, episodes not stored; accumulated (the
                                   caller zeroes it) */
  int64_t cap_polys, cap_terms;
} bb_poly_sink;

/* bb_run_export: bb_run (same arguments, same order, same records) that also writes polynomials of every episode into
 * caller-owned device sinks -- the first return value of buchberger(), interreduce(minimalize(G)) (buchberger.cpp:265),
 * for a whole batch of episodes.  bb_run is bb_run_export with both sinks NULL.
 *   gb     (may be NULL; needs compute_gb != 0): the reduced Groebner basis of every episode that ends BB_STATUS_DONE,
 *          ascending lead monomial, monic -- what bb_final_gb returns for that episode.
 *   basis  (may be NULL): the final basis G of every episode that ends BB_STATUS_DONE or is cut by max_steps (its record
 *          keeps BB_STATUS_RUNNING), in insertion order -- what bb_download_basis returns.
 * An episode that ends in any other status (an overflow, or BB_STATUS_OVERFLOW_SCRATCH while interreducing) stores nothing.
 * where_dev is indexed by the call's episode index e = 0 .. episodes-1, across the 65536-episode batches of one call.
 * Space is reserved per episode by atomics on used_dev[0..1], so where in the buffers an episode lands depends on the order
 * in which episodes finish; the contents and lengths stored for an episode do not.  An episode that does not fit gets
 * where = (-1, -1) and increments used_dev[2]; its reservation still counts, so after the call used_dev[0..1] are the
 * exact capacities that store every episode.  Episode records and statuses are bit-identical with and without sinks.
 * The sinks are captured by the call: calls in flight on different streams need their own.  Fails (nothing enqueued) for a
 * gb sink with compute_gb == 0, and for a sink with a NULL buffer or a negative capacity; the size of where_dev is the
 * caller's to get right. */
int bb_run_export(bb_handle* h, int strategy, int episodes, int seed_base, const int32_t* seeds_dev, int sel_seed_base,
                  int max_steps, double gamma, int compute_gb, bb_episode_stats* stats_dev, int32_t* trace_dev,
                  int trace_episodes, int trace_cap, void* stream, const bb_poly_sink* gb, const bb_poly_sink* basis);

/* bb_reduce: the division algorithm reduce(g, F) (buchberger.cpp:24-49) for a batch of dividends against caller-supplied
 * divisor lists, on the device.  While h != 0: the first f of F (scanned in order) with LM f | LM h gives
 * h <- h - (LT h / LT f) f and steps += 1; otherwise LT h moves to the remainder.  The remainder is not made monic.
 *   divisor lists   exactly the layout of a run_episodes(return_gb) batch: list_offsets_dev int64 [nlists + 1] indexes
 *                   polynomials, poly_offsets_dev int64 [npolys + 1] indexes terms, exps_dev int32 [nterms * n],
 *                   coefs_dev int32 [nterms]; n = cfg.nvars
 *   queries         q_offsets_dev int64 [nqueries + 1] into q_exps_dev / q_coefs_dev (same term layout); query q is reduced by
 *                   list which_dev[q].  Queries that share a list should be adjacent: a worker restages a list only when
 *                   it changes.
 * Every polynomial has its terms strictly descending in grevlex with coefficients in [1, p).  sorted = 0 scans each list in
 * the order given; sorted = 1 scans it stable-sorted by ascending lead monomial (the order of G_ under sort_reducers,
 * buchberger.cpp:308-311), which lets the scan stop early; a reduced basis from bb_run_export is already in that order.
 * Outputs per query: steps_dev, rlen_dev (remainder length) and status_dev, all int32 [nqueries].  Status BB_STATUS_DONE, or
 *   BB_STATUS_OVERFLOW_EXPONENT  an exponent above the packed layout's field, or a produced monomial that leaves it
 *   BB_STATUS_OVERFLOW_SCRATCH   a dividend longer than cfg.max_poly_terms (also while reducing)
 *   BB_STATUS_OVERFLOW_BASIS     a list longer than cfg.max_basis
 *   BB_STATUS_OVERFLOW_TERMS     the list plus the remainder do not fit cfg.max_terms
 *   -1                           malformed input: terms not strictly descending, a coefficient outside [1, p), a negative
 *                                exponent, a zero polynomial in a list, bad offsets, which outside [0, nlists)
 * A query that does not end done gets steps = rlen = 0 and stores nothing.  rem (may be NULL: lengths, steps and status only,
 * e.g. for ideal membership) receives the remainder of every query that ends done as entry q, one polynomial, with where_dev
 * [nqueries * 2] and used_dev behaving as in bb_run_export (after the call used_dev[0..1] hold the exact totals).
 * bb_counters: additions += sum of steps; terms_read, terms_written, lms_scanned and term_moves (= sum of rlen) as for the
 * episodes, over the queries that end done; env_steps and episodes do not change.
 * Fails with nothing enqueued for a negative count, a NULL required pointer, or a sink with a NULL buffer or a negative
 * capacity.  The call takes a bank of environment slots by the rule of bb_run (see "Pipelines" below): like bb_run, a call on
 * the stream the step API uses overwrites the step API's environments. */
int bb_reduce(bb_handle* h, int nlists, const int64_t* list_offsets_dev, const int64_t* poly_offsets_dev,
              const int32_t* exps_dev, const int32_t* coefs_dev, int nqueries, const int64_t* q_offsets_dev,
              const int32_t* q_exps_dev, const int32_t* q_coefs_dev, const int32_t* which_dev, int sorted, int32_t* steps_dev,
              int32_t* rlen_dev, int32_t* status_dev, const bb_poly_sink* rem, void* stream);

/* Pipelines.  Calls of bb_run on ONE stream run one after the other in the handle's own environments.  A call on a second
 * stream while a runner of the first is still at work uses another bank of environment slots (up to three banks, each
 * allocated on first use; a fourth concurrent call queues behind the least recently started one), so the runners of
 * consecutive batches overlap: the CTAs of batch i + 1 move in while batch i drains (an episode runner ends with its longest
 * episodes on a mostly idle GPU).  Host views (bb_download_basis, bb_final_gb, bb_stats ...) read the first bank.
 *
 * bb_prepare: the preparation half of the NEXT bb_run call (ideal generator + reset() of every episode of the batch,
 * buchberger.cpp:299-315) enqueued on `stream`, which may be a different stream than the one the runner uses: the handle
 * keeps a ring of three staging sets, so batches can be prepared up to two calls ahead of the runner.  A later bb_run
 * with the same (episodes, seed_base, seeds_dev) takes the oldest such batch instead of preparing; any other bb_run ignores it.
 * episodes <= 65536 (one batch).  Results are those of bb_run alone. */
int bb_prepare(bb_handle* h, int episodes, int seed_base, const int32_t* seeds_dev, void* stream);

/* bb_set_episode_offset: global index of episode 0 of the following bb_run calls (default 0).  Episode e of a call then
 * seeds its Random-selection stream with sel_seed_base + (offset + e) * stride and replays staged ideal
 * (offset + e) mod staged count -- a rank that runs episodes [first, first + count) of a job gets the records of that
 * slice of the whole job (sharding.py).  The ideal stream is still seeded seed_base + e (or seeds_dev[e]). */
int bb_set_episode_offset(bb_handle* h, int offset);

/* bb_set_timing / bb_last_run_ms: with timing on, bb_run records CUDA events on its stream around the preparation and
 * around the episode runner of its first batch; bb_last_run_ms synchronises on them and returns both durations (bench.py:
 * the roofline of the runner kernel on its own launch time). */
int bb_set_timing(bb_handle* h, int on);
int bb_last_run_ms(bb_handle* h, float* prepare_ms, float* run_ms);

/* bb_set_selection_seed_stride: bb_run seeds episode e's BB_SELECT_RANDOM stream with sel_seed_base + e * stride.
 * Default 1 (every episode its own stream); 0 gives every episode the SAME seed, which is what scripts/make_strat.cpp:66
 * does (one `seed` argument for every ideal of the file). */
int bb_set_selection_seed_stride(bb_handle* h, int stride);

/* bb_set_prepare_mode: how bb_run prepares a batch of episodes (ideal generator + reset(), buchberger.cpp:299-315).
 * 0 (default): one THREAD per episode where it applies (binomial distributions with at most 16 generators), else one
 * warp per episode; 1: always one warp per episode.  Both produce bit-identical states and counters; this is a
 * performance switch that the tests use to compare the two. */
int bb_set_prepare_mode(bb_handle* h, int by_warp);

/* bb_set_two_term: which warp runner bb_run uses for binomial distributions (bb_set_distribution), whose polynomials all
 * have at most two terms.  1 (default): a runner built for that case (register-only arithmetic, the remainder handed to
 * update() in registers); 0: the general runner.  Both produce bit-identical records, counters and exported polynomials;
 * this is a performance switch that the tests use to compare the two.  Other ideals always use the general runner. */
int bb_set_two_term(bb_handle* h, int on);

/* bb_set_wide: how bb_run's episode runner reduces.  0: the dividend is materialised (warp-cooperative merges, built
 * for the 2-term polynomials of binomial ideals); 1: the dividend is a set of streams into the term arena, one round per
 * lead term and O(1) work per addition (built for long polynomials, e.g. cyclic-n), run by one CTA per environment
 * (shortest chain of additions: a cyclic-6 launch lasts as long as its longest episode; 256 streams in registers, 768
 * more in shared memory); -1 (default): 1 when the capacities are sized for long polynomials (max_poly_terms >= 256),
 * else 0.  Test modes: 2 / 3 as 1 with 6 / 48 stream slots (consolidation of the dividend into a scratch list every few
 * additions); 7 as 1 with 8 register slots (the shared-memory table on every step); 8 as 1 with 32 instead of 256
 * reducers in the control warp's registers (the rest of the reducer list scanned in memory).  Modes 4, 5 and 6 are kept
 * for compatibility and are the same as 1, 2 and 3.  Every mode produces bit-identical episodes; this is a performance
 * switch.  Of the bb_counters, terms_read / terms_written count |h| per addition only where h is materialised
 * (mode 0). */
int bb_set_wide(bb_handle* h, int mode);

/* bb_value: BuchbergerEnv::value(strategy, gamma) (buchberger.cpp:332-351) for every environment at once:
 * value_dev double[N] = discounted return of finishing the episode from the CURRENT state under `strategy`
 * (0.0 for an environment that is not running).  The environments are forked into a private arena; their own state
 * is untouched.  strategy = BB_SELECT_RANDOM runs `rollouts` rollouts per environment (stream seeds sel_seed_base + r)
 * and keeps the best; BB_VALUE_SAMPLE is value("sample"): one Degree rollout and rollouts-1 (default 100) Random
 * rollouts seeded sel_seed_base + 0..99, best kept (:333-341; the reference seeds these from std::random_device).
 * A rollout that overflows an arena yields NaN for its environment.  bb_rollout_value computes the same value for every
 * state of a fused rollout. */
int bb_value(bb_handle* h, int strategy, double gamma, int rollouts, int sel_seed_base, int max_steps,
             double* value_dev, void* stream);

/* bb_copy_env: the copy constructor (buchberger.cpp:279-283; copy() of wrapped.pyx:35-38): environment src_env of
 * `src` -> environment dst_env of `dst`, including both random streams and the staged ideal.  The handles must be on
 * the same device with equal nvars, prime and capacities (they may be the same handle). */
int bb_copy_env(bb_handle* dst, int dst_env, bb_handle* src, int src_env, void* stream);

/* ---- vector-environment conveniences
 * bb_set_auto_reset(on): with on != 0, bb_step and bb_rollout reset an environment in the same call in which it
 * finishes: the caller sees done = 1 for that transition and the first state of the NEXT episode (drawn from the
 * environment's own ideal stream) afterwards -- the loop of pg.Agent.run_episodes (pg.py:477-503) without a host
 * round trip, and no idle slots. */
int bb_set_auto_reset(bb_handle* h, int on);

/* bb_set_prefetch: a reset inside a step kernel (auto-reset) is one warp's detour through the ideal generator and s update()
 * calls -- 38 us during which the rest of the launch waits for that warp.  With prefetch every environment keeps a queue of
 * `depth` initial states of its NEXT episodes, prepared in bulk from the environment's own ideal stream (in stream order: what
 * an environment draws is unchanged) by one thread per environment; bb_reset / auto-reset then take the head of the queue with
 * a copy, and bb_step / bb_step_observe top the queues up every 4 * depth calls, bb_reset and bb_rollout at every call.  Applies
 * to binomial distributions with at most 16 generators.  depth 0 turns it off; default 8 for handles of at least 64
 * environments.  bb_seed, bb_copy_env and a change of the distribution drop the queues concerned. */
int bb_set_prefetch(bb_handle* h, int depth);

/* bb_set_max_episode_length: bb_step / bb_step_observe / bb_step_host / bb_rollout cut an episode once it has MORE than
 * `max_steps` steps (the loop of pg.Agent.run_episode, pg.py:470-471: `if episode_length > max_episode_length: break`;
 * train.py's default is 500): the environment goes to BB_STATUS_TRUNCATED, reports done = 1 and is reset by auto-reset
 * like a finished one.  0 (default) = unlimited. */
int bb_set_max_episode_length(bb_handle* h, int max_steps);

/* ---- batch management (north_star: "finished or diverged episodes are compacted by stream compaction")
 * bb_compact: active_dev int32[N + 1] <- (number of RUNNING environments, then every slot with the RUNNING ones first,
 * both groups ascending); active_dev == NULL refreshes the handle's own list only.  bb_step / bb_step_observe /
 * bb_step_host run it themselves when auto-reset is off (bb_set_compaction(0) turns that off) and take the environments
 * in that order, so stepping warps fill whole CTAs; results are identical either way.
 * bb_status_summary: counts_host int32[BB_STATUS_COUNT] <- number of environments per BB_STATUS_* word (finished,
 * truncated and diverged = every BB_STATUS_OVERFLOW_* / BAD_ACTION); synchronises the stream. */
int bb_set_compaction(bb_handle* h, int on);
int bb_compact(bb_handle* h, int32_t* active_dev, void* stream);
int bb_status_summary(bb_handle* h, int32_t* counts_host, void* stream);

/* bb_set_obs_nvars: state matrices show only the first n_obs variables of every monomial (cols = 2 * n_obs * k).  This
 * exists for byte-level comparison with the reference's C++ / Cython LeadMonomialsEnv on FIXED ideals, whose
 * FixedIdealGenerator::nvars is the largest variable INDEX in use, i.e. one less than the number of variables
 * (ideals.cpp:146-154): cyclic-6 is observed with n = 5, 20 columns.  The default follows the Python environment
 * (ring.ngens, buchberger.py:537).  Episodes are not affected; the policy head is not available in this mode. */
int bb_set_obs_nvars(bb_handle* h, int n_obs);

/* ---- the pairs policy head on device (SURVEY 8 a15)
 * bb_policy_pmlp: ParallelMultilayerPerceptron([hidden]) (networks.py:522-571) evaluated on every environment's
 * current state matrix, then tf.random.categorical (pg.py:323-326):
 *     logit[r] = b2 + sum_u w2[u] * relu(b1[u] + sum_c W1[c*hidden + u] * state[r][c])        (fp32)
 *     logp = log_softmax(logit over the |P| rows);  action = first row whose inclusive prefix sum of
 *     exp(logit - max) exceeds u * total, u = (bb_hash_item(seed + env, counter) >> 40) * 2^-24   (greedy: argmax)
 * The first layer runs on the tensor cores (TF32 MMA with W1 split into two TF32 halves, exact integer inputs, fp32
 * accumulation): logits agree with an fp32 evaluation to ~1e-6 relative (tests: rtol = atol = 1e-5 against torch fp32).
 * W1 is [cols, hidden] row-major (the Keras Dense kernel), b1 [hidden], w2 [hidden] (Dense(1) kernel), b2 [1];
 * hidden in {32, 64, 128, 256}.  actions_dev int32[N] (0 for environments that are not running), logprob_dev
 * float[N] = logp[action] (optional), logprobs_all_dev float[N, pmax] (optional; rows >= |P| untouched). */
int bb_policy_pmlp(bb_handle* h, int hidden, const float* W1_dev, const float* b1_dev, const float* w2_dev,
                   const float* b2_dev, uint64_t seed, uint64_t counter, int greedy, int32_t* actions_dev,
                   float* logprob_dev, float* logprobs_all_dev, int pmax, void* stream);

/* bb_rollout: T steps of every environment in ONE launch -- policy head, sample, step, auto-reset (if enabled) --
 * i.e. the loop of pg.Agent.run_episode (pg.py:451-472) fused on device.  Step t of environment e draws its uniform
 * with counter counter0 + t.  Outputs are environment-major [N, T] (any may be NULL): actions (-1 where the
 * environment was not running), logprob, reward (float: -(additions) or -1), done, lengths (|P| before the step);
 * obs_dev (optional) int32 [N, T, pmax, cols] = the state matrix before each step, padded with -1 (pg.py:217-226). */
int bb_rollout(bb_handle* h, int hidden, const float* W1_dev, const float* b1_dev, const float* w2_dev, const float* b2_dev,
               uint64_t seed, uint64_t counter0, int greedy, int T, int32_t* actions_dev, float* logprob_dev,
               float* reward_dev, uint8_t* done_dev, int32_t* lengths_dev, int32_t* obs_dev, int pmax, void* stream);

/* bb_rollout_value: bb_rollout that also writes value_dev double [N, T] (environment-major): value[e][t] = bb_value of the
 * state step t of environment e starts from (the state obs[e][t] shows, with |P| = lengths[e][t]), i.e. the baseline
 * pg.Agent.run_episode stores when the agent has a value model 'degree' / 'sample' (pg.py:461-462), computed inside the
 * same launch; 0.0 where the environment is not running.  value_strategy, value_gamma, value_rollouts, value_sel_seed and
 * value_max_steps are bb_value's strategy, gamma, rollouts, sel_seed_base and max_steps, with bb_value's rules (seeds,
 * rollout counts, NaN for a rollout that overflows an arena); pass bb_value the gamma of the advantages (pg.py passes its
 * own gam).  So with auto-reset on, the loop
 *     for t in 0..T-1:  bb_value(v[:, t]); bb_policy_pmlp(counter0 + t); bb_step
 * gives bit-identical values, actions, log-probabilities, rewards, done flags and lengths.  Everything else bb_rollout
 * writes -- outputs, the environments after the call, their random streams and prefetch queues, bb_stats and
 * bb_counters -- is identical to bb_rollout with the same arguments: the value rollouts run in a fork arena of one slot
 * per environment (kept with bb_value's, 8 GiB at most) and their traffic is not counted.  The rollouts of one state run
 * one after another in that environment's warp, so 'sample' (101 rollouts) costs about 101 times 'degree' per step.
 * value_dev == NULL is bb_rollout (the value arguments are still checked).  Fails (nothing enqueued) for what bb_rollout
 * refuses, a bad value strategy, and a fork arena that cannot be allocated or would exceed 8 GiB. */
int bb_rollout_value(bb_handle* h, int hidden, const float* W1_dev, const float* b1_dev, const float* w2_dev,
                     const float* b2_dev, uint64_t seed, uint64_t counter0, int greedy, int T, int32_t* actions_dev,
                     float* logprob_dev, float* reward_dev, uint8_t* done_dev, int32_t* lengths_dev, int32_t* obs_dev, int pmax,
                     int value_strategy, double value_gamma, int value_rollouts, int value_sel_seed, int value_max_steps,
                     double* value_dev, void* stream);

/* bb_rollout_rows: bb_rollout_value (value_dev may be NULL) that also stores the state matrix of every step at its own
 * row count -- the reference's TrajectoryBuffer, which keeps each state unpadded and pads only when it forms a batch
 * (pg.py:162-241) -- so no state is lost to a pmax.  rows_dev int32 [N, rows_per_env, cols]: environment e owns rows
 * rows_dev[e][0 .. rows_per_env) (of which one call fills at most 2^31 - 1).  The |P| = lengths[e][t] rows of each state an action is taken from (actions[e][t] >= 0)
 * go there back to back, in step order, without padding; rows past the last state are untouched.  So the rows of step t
 * start at row  sum of lengths[e][t'] over t' < t with actions[e][t'] >= 0  of e's region.
 * Budget rule: when the rows of the state step t of environment e starts from do not fit into what is left of e's region,
 * e takes no further step in this call: steps t..T-1 get action -1, logprob 0, reward 0, done 0, lengths 0, value 0.0 and
 * obs all -1, and e keeps the state of step t, so the next call continues it and no state is lost.  This is the only way
 * an output has action -1 with done 0 (a slot that is not running reports done 1).  Halted steps are not env-steps;
 * bb_counters' obs_rows counts the rows written (row store and obs).  Every step before the halt is exactly what the same
 * call without a row store gives (step t still samples with counter counter0 + t).  rows_dev and obs_dev are independent.
 * rows_dev == NULL is bb_rollout_value.  Fails (nothing enqueued) for what bb_rollout_value refuses, and for rows_dev !=
 * NULL with rows_per_env < bb_config.max_pairs: that minimum lets every environment store the state it starts from. */
int bb_rollout_rows(bb_handle* h, int hidden, const float* W1_dev, const float* b1_dev, const float* w2_dev,
                    const float* b2_dev, uint64_t seed, uint64_t counter0, int greedy, int T, int32_t* actions_dev,
                    float* logprob_dev, float* reward_dev, uint8_t* done_dev, int32_t* lengths_dev, int32_t* obs_dev, int pmax,
                    int value_strategy, double value_gamma, int value_rollouts, int value_sel_seed, int value_max_steps,
                    double* value_dev, int32_t* rows_dev, int64_t rows_per_env, void* stream);

/* bb_run_policy: bb_run_export with the PMLP head of bb_policy_pmlp choosing every pair instead of a SelectionType -- the
 * trained agent evaluated on whole episodes (pg.Agent.run_episode, pg.py:451-472, run to completion), with the same
 * records, traces, sinks, batching, bb_prepare matching, banks, max_steps truncation and bb_counters as bb_run_export.
 * Weights, hidden and greedy are those of bb_policy_pmlp (greedy: argmax, the lowest row on ties).  Step t of episode e of
 * the call draws its uniform from stream seed + (offset + e) and counter counter0 + t, where offset is bb_set_episode_offset's
 * value: a record depends only on the episode's global index, never on the slot, the handle's size, the batching or the
 * sharding.  So environment e of the step API, seeded seed_base + e and driven by bb_policy_pmlp(seed, counter0 + t) + bb_step
 * at its step t, plays exactly episode e of bb_run_policy(seed, counter0, ..., seed_base).  Every step uses the
 * materialising reduction, whatever bb_set_wide and bb_set_two_term say (identical episodes).  Fails (nothing enqueued) for
 * what bb_policy_pmlp refuses, episodes < 0, stats_dev == NULL, a gb sink with compute_gb == 0, and a bad sink. */
int bb_run_policy(bb_handle* h, int hidden, const float* W1_dev, const float* b1_dev, const float* w2_dev,
                  const float* b2_dev, uint64_t seed, uint64_t counter0, int greedy,
                  int episodes, int seed_base, const int32_t* seeds_dev, int max_steps, double gamma, int compute_gb,
                  bb_episode_stats* stats_dev, int32_t* trace_dev, int trace_episodes, int trace_cap, void* stream,
                  const bb_poly_sink* gb, const bb_poly_sink* basis);

/* bb_discount: discounted suffix sums inside episode segments, the primitive of pg.discount_rewards (pg.py:18-39) and
 * of the generalised advantage estimates (pg.compute_advantages, pg.py:42-78) on the [N, T] trajectories bb_rollout
 * writes:  out[n][t] = x[n][t] + (done[n][t] ? 0 : gam * out[n][t+1]),  out[n][T] = 0, in fp64 (mul then add, no fma). */
int bb_discount(bb_handle* h, int N, int T, const double* x_dev, const uint8_t* done_dev, double gam, double* out_dev,
                void* stream);

/* ---- host views (synchronising)
 * bb_download_basis: basis G of environment env in insertion order: lens[npoly], exps[nterms*n], coefs[nterms].
 * Returns the number of polynomials, or <0; *nterms_out receives the number of terms. */
int bb_download_basis(bb_handle* h, int env, int32_t* lens, int cap_polys, int32_t* exps, int32_t* coefs,
                      int cap_terms, int* nterms_out);
/* bb_final_gb: interreduce(minimalize(G)) (buchberger.cpp:102-122, 265) of environment env computed ON DEVICE,
 * ascending lead monomial, monic.  Same output convention as bb_download_basis. */
int bb_final_gb(bb_handle* h, int env, int32_t* lens, int cap_polys, int32_t* exps, int32_t* coefs, int cap_terms,
                int* nterms_out);
int bb_counters_read(bb_handle* h, bb_counters* out, int reset);

/* ---- checksums (so a host-side checker can recompute them from an oracle's episode)
 * item(x, pos) = splitmix64_finalizer(x + 0x9E3779B97F4A7C15 * (pos + 1));  all sums are mod 2^64.
 *   trace_hash = h_T, where h_0 = 0 and h_{t+1} = h_t * 0x9E3779B97F4A7C15 + (i | j<<16 | additions<<32) + 1 over the
 *        steps in order (a rolling polynomial hash: one multiply-add per step on the device)
 *   basis_hash / gb_hash = sum over terms t (flattened over the polynomial list, in order) of
 *        item(coef, 3t) + item(e0 | e1<<16 | e2<<32 | e3<<48, 3t+1) + item(e4 | e5<<16 | e6<<32 | e7<<48, 3t+2)
 *      + sum over polynomials q of splitmix64_finalizer(len_q + 0xD1B54A32D192ED03 * (q + 1)) */
uint64_t bb_hash_item(uint64_t x, uint64_t pos);

#ifdef __cplusplus
}
#endif
#endif /* BBENV_H */
