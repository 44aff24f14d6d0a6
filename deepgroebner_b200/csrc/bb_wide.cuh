// bb_wide.cuh -- reduce() for LONG polynomials (cyclic-n and other non-binomial ideals, BASELINE configs[4]) without
// ever materialising the dividend, run by a whole CTA (BBW_WARPS warps) on ONE environment, sm_100a.
//
// warp_reduce / warp_merge (bb_device.cuh) are built for binomial ideals, where a polynomial is two terms.  On cyclic-6
// (SURVEY 8 a4/a6) a dividend of ~100 (up to ~550) terms is reduced ~83 times per step by polynomials of ~37 terms, and an
// episode is a serial chain of ~80 000 such additions (697 000 in the longest of 1024): materialising
// h <- h - (LT h / LT f) f (buchberger.cpp:33-35) costs O(|h| + |f|) work per addition and, whatever the parallel merge,
// several dependent passes over memory.  Round 2 built and measured three block-wide merges for it (merge path, a
// two-barrier bitmap merge, streams with one barrier per lead term: 1.85 / 1.5 / 1.5 us per addition) before settling on:
//
//   h = sum over STREAMS i of  nc_i * m_i * tail(f_i)        (the S-polynomial's two halves, then one stream per addition)
//
// A stream is a cursor into the term arena plus its multiplier; its current term (scaled) is its HEAD.  The lead term of
// h is the smallest head key (keys ascend as monomials descend) with the SUM of the coefficients of every head that
// carries it; a zero sum is a cancelled monomial and is skipped.  This is the division algorithm of buchberger.cpp:24-49
// with Polynomial operator+ (polynomials.cpp:148-177) evaluated lazily: the sequence of lead terms, the reducer chosen
// for each (first in G_ whose lead monomial divides), the number of additions (the reward) and the remainder are those
// of the reference, term for term and bit for bit -- only the order in which coefficients are summed differs, and
// addition mod p is associative.  An addition costs O(1) and each term of a reducer is touched once.
//
// One ROUND per lead term M: (a) M's first divisor among the reducer lead monomials (buchberger.cpp:27-32), (b) every
// stream whose head is M advances -- the next raw term was prefetched into registers a round earlier -- and each thread
// takes the minimum over its heads with the coefficient sum at it, (c) REDUX reductions give the next lead term.  A divisor
// f opens a new stream whose head comes straight from f's head record (no dependent load).  Measured on the longest
// cyclic-6 episode (697 000 additions): 955 000 rounds (73 % additions, 21 % remainder terms, 6 % cancelled monomials)
// for 26 M stream terms, i.e. ~27 streams advance per round and a few hundred are live: the monomials of h and of the
// reducers' multiples coincide massively, which is why h stays short while the streams are many.
//
// A stream slot is free when its head key is all ones; a new stream takes a free slot, so the tables stay as small as the
// number of LIVE streams.  If no slot is free, h is consolidated: every pending term is written in order to a scratch list
// behind the slot's term arena and h goes on as ONE stream over it (bb_set_wide(2 / 3) cap the slots so that the tests
// reach this).
//
// Episode records are bit-identical to the materialising runner's (bb_set_wide(0): warp_merge / warp_reduce, an
// independent second implementation); of the traffic counters, terms_read / terms_written (|h| per addition) are not
// observable without materialising h and count the reducers' lengths only.
//
// A cyclic-6 launch is as long as its longest episode (697 000 dependent additions in the longest of 1024 seeded-Random
// episodes), so what decides it is the latency of one ROUND (one lead monomial of the dividend: its coefficient, its
// divisor, the advance of the streams that carry it, the next lead monomial).  A round is a dependent chain of
// instructions, issued one per ~4 cycles, plus fixed latencies (measured on B200, tools/ub/lat.cu: REDUX.MIN 22 cycles,
// REDUX.ADD 47 -- a warp's REDUX operations do not overlap --, STS + BAR + LDS 58), so the CTA is WARP-SPECIALISED to keep
// every warp's chain short:
//   * the first BBW_WARPS - 1 warps are STREAM warps: thread t owns the stream in REGISTER slot t; in a round it adds its
//     head's coefficient to the round's sum and advances if its head is the lead monomial, and the warp folds its minimum
//     head key (two REDUX), coefficient sum (one) and first free slot (a ballot) into a 16-byte record;
//   * the last warp is the CONTROL warp: 256 reducer lead monomials of G_ (and their basis indices) in its registers; in a
//     round it finds the lead monomial's first divisor, loads the divisor's head record and writes everything about the
//     stream this divisor opens that does not depend on the coefficient -- head key, multiplier monomial, term range,
//     counter increments -- as a 48-byte descriptor to shared memory;
//   * ONE block barrier per round; behind it every warp folds the stream warps' records (one per lane) and reads the
//     descriptor; the thread that owns the new stream's slot alone works out the multiplier and head coefficients; one
//     warp keeps the reduction's books (remainder, counters, sugar) and publishes them at the end.
// Longest episode: 0.79 us per addition (1.37 rounds); clock probes (-DBBW_CLOCK) give per round ~480 cycles before the
// barrier for the control warp (330 - 450 for the stream warps), ~300 for barrier + fold, ~230 - 300 behind it.
//
// A new stream takes the first free register slot of the block (the fold reports it), so the register slots hold the LIVE
// streams; only when all BBW_SLOTS are live does a stream go to the shared-memory table behind them (append only;
// scanned by its owner thread each round), and only when that is full too is h consolidated (see above).
// bb_set_wide(2 / 3): 6 / 48 register slots and no table (consolidations every few additions); bb_set_wide(7): 8 register
// slots and the whole table (the shared-memory path on every step); bb_set_wide(8): the control warp keeps 32 reducers in
// registers instead of 256 (its scan of the rest of G_ in memory on most rounds).
//
// Every routine that touches the per-thread state is inlined: a call would take the state's address and move it from
// registers to local memory (LDL / STL on the chain of every round: 1.35 -> 1.06 us per addition when that was removed).
#pragma once
#include "bb_device.cuh"

#ifndef BBS_KMAX
#define BBS_KMAX 1024           // BBRunArgs::stream_kmax when bb_set_wide does not cap the streams
#endif
#define BBS_NONE 0xffffffffu

// The scratch list of a consolidation lies BEHIND the term arena of the slot (bbenv.cu lays hkey right after tkey and
// hcoef right after tcoef, max_terms a multiple of 8), so term index max_terms + i addresses scratch term i through the
// same two base pointers and a stream's cursor needs no flag.  Two halves of max_poly_terms terms: a consolidation writes
// one while the stream over the other is still being read.

__device__ __forceinline__ uint32_t bbf_reduce(const BBField& F, uint32_t x) {   // x mod p for any x < 2^32
  const uint32_t q = __umulhi(x, F.mu);
  const uint32_t r = x - q * F.p;
  return r >= F.p ? r - F.p : r;
}

#ifndef BBW_WARPS
#define BBW_WARPS 8
#endif
#define BBW_THREADS (BBW_WARPS * 32)
#ifndef BBW_MIN_CTAS
#define BBW_MIN_CTAS 2
#endif
#ifndef BBW_KMAX
#define BBW_KMAX 1024           // BBW_KMAX - BBW_THREADS entries in the shared-memory table behind the register slots
#endif
static_assert(BBW_KMAX % BBW_THREADS == 0 && BBW_KMAX > BBW_THREADS, "whole rows of streams");
static_assert(BBW_WARPS <= 32 && (BBW_WARPS & (BBW_WARPS - 1)) == 0, "one record per lane in the folds; a power of two (block_add_basis)");
static_assert(BBW_KMAX / BBW_THREADS <= 8, "per-thread coefficient sums of a round stay below 2^19, a warp's below 2^24");
#define BBW_NOFREE 0x3fu

struct WideStreams {             // dynamic shared memory: the table behind the register slots (entry i belongs to thread i % BBW_THREADS)
  uint64_t key[BBW_KMAX - BBW_THREADS];
  uint64_t adj[BBW_KMAX - BBW_THREADS];
  uint64_t pkey[BBW_KMAX - BBW_THREADS];
  uint32_t coef[BBW_KMAX - BBW_THREADS];
  uint32_t nc[BBW_KMAX - BBW_THREADS];
  uint32_t pcoef[BBW_KMAX - BBW_THREADS];
  uint32_t ptr[BBW_KMAX - BBW_THREADS];
  uint32_t end[BBW_KMAX - BBW_THREADS];
};

#define BBW_SLOTS ((BBW_WARPS - 1) * 32)   // register slots = stream threads: the last warp of the block is the CONTROL warp

#ifdef BBW_CLOCK
__device__ __forceinline__ long long bbw_clock(uint32_t dep) {   // the clock, read once `dep` has been computed
  long long t;
  asm volatile("mov.u64 %0, %%clock64;" : "=l"(t) : "r"(dep) : "memory");
  return t;
}
#endif

struct WideShared {
  // per-warp round results of the stream warps, double-buffered: (min head key lo, hi, coefficient sum of the consumed
  // monomial | first free lane << 24, -)
  __align__(16) uint4 wrec[2][BBW_WARPS];
  // what the control warp found for the round's lead monomial M, double-buffered: [0] = (key of the new stream's head
  // f.k1 + M - f.lm lo, hi, key(M / LM f) - bias lo, hi), [1] = (f.invlc | f.c1 << 16, first term behind the head, end,
  // flags: 1 a divisor exists, 2 the head key overflowed its exponent fields), [2] = (lead monomials scanned: the
  // counter's increment, the sugar f would give the result, -, -)
  __align__(16) uint4 desc[2][3];
  // what the book-keeping warp kept count of during a reduction, published at its end: (remainder length or -BB_STATUS_*,
  // reductions, sugar of the result, -), (lead monomials scanned, reducer terms read, terms moved to the remainder, -)
  __align__(16) uint4 fin[2];
  int row;                  // the pair row warp 0 selected
  long long upd;            // result of warp_add_basis
  // block_add_basis: per-warp results of one sweep of the peeling loop, double-buffered: (largest undecided key lo, hi,
  // its lowest index, a member of the current kept lcm's group is coprime to the new element)
  __align__(16) uint4 prec[2][BBW_WARPS];
};

// Block-uniform state of a step's reduction plus per-thread registers; every member is a scalar so that the whole record
// lives in registers.
struct WideState {
  int T;                    // entries of the shared-memory table in use (append only until a consolidation)
  int tcap;                 // entries of the table that may be used
  int regs;                 // register slots that may be used (threads 0 .. regs - 1), at most BBW_SLOTS
  int cbase;                // reducers of G_ the control warp keeps in registers (256; 32 under bb_set_wide(8)): the rest is scanned in memory
  int cz;                   // scratch half the next consolidation writes
  // stream threads: the stream in this thread's register slot.  k0 all ones: free.
  uint64_t k0, adj0, pk0; uint32_t c0, nc0, pc0, p0, e0;
  // control warp: reducers lane, lane + 32, ... lane + 224 of G_: the exponent fields of the lead monomial and
  // (position << 16) | basis index (BBS_NONE: absent)
  uint64_t rl[8]; uint32_t rc[8];
  // stream threads: the raw term behind the head of table entry pend_i, loaded but not yet stored to st.pkey / st.pcoef
  int pend_i; uint64_t pend_k; uint32_t pend_c;
  uint32_t bad;             // per thread: a produced key overflowed its exponent fields
#ifdef BBW_INSTR
  long long n_rounds, n_trounds, sum_T, n_consol, n_crounds, n_topen;   // diagnostic counts (block-uniform)
#endif
#ifdef BBW_CLOCK
  long long s_sel, s_take, s_red, s_upd;   // diagnostic: cycles of a step's parts (select, pair removal, reduction, update)
  long long cw, cb, cp, co, tl; // diagnostic: cycles before the round's barrier, barrier + fold, post-processing, outside; end of the last post-processing
#endif
  __device__ __forceinline__ void clear() {
    T = 0; k0 = ~0ull; adj0 = pk0 = 0ull; c0 = nc0 = pc0 = p0 = e0 = 0u; pend_i = -1; pend_k = 0ull; pend_c = 0u; bad = 0u;
  }
};

// One round by the block for the lead monomial M of h (M all ones, the pseudo lead monomial a reduction starts from:
// nothing is consumed, S is meaningless).
//   stream warps: S = the sum of the coefficients of the heads that carry M (taken HERE, when M is consumed, so that the
//     sum's reduction is off the chain of the 64-bit minimum), those streams advance, M2 = the minimum head key after that
//     (all ones: h is exhausted), freet = the first thread whose register slot is free (-1: none);
//   control warp, concurrently (search): M's first divisor f in G_ (buchberger.cpp:27-32), f's head record, and everything
//     about the stream f would open that does not depend on S, as the round's descriptor (dA, dB; see WideShared).
// One barrier; behind it every warp folds the stream warps' records and reads the descriptor.  `half` = which half of the
// double buffers this round uses.
template <int NV>
__device__ __forceinline__ void wide_round(WideShared& sh, int& half, WideState& ws, WideStreams& st, const BBField F,
                                           const uint64_t M, const bool search, const GHeadMem* gh, const uint64_t* rlm,
                                           const uint32_t* ridx, const int nR, const bool sorted, const uint64_t* tk,
                                           const uint32_t* tc, uint32_t& S, uint64_t& M2, uint4& dA, uint4& dB, uint4& dC, int& freet) {
  typedef KL<NV> K;
  const int tid = threadIdx.x, lane = bb_lane();
#ifdef BBW_INSTR
  ws.n_rounds++; if (ws.T > 0) { ws.n_trounds++; ws.sum_T += ws.T; } if (!search) ws.n_crounds++;
#endif
#ifdef BBW_CLOCK
  const long long t0 = bbw_clock((uint32_t)M);
  ws.co += t0 - ws.tl;
#endif
  if (tid >= BBW_SLOTS) {
    // ---- control warp: the divisor search and the head record of the divisor
    if (search && M != ~0ull) {
      const uint64_t mg = (M & K::ex_mask) | K::ge_mask;
      uint32_t cand = BBS_NONE;
#pragma unroll
      for (int q = 7; q >= 0; q--)
        if (((mg - ws.rl[q]) & K::ge_mask) == K::ge_mask) cand = ws.rc[q];   // rl: exponent fields only; absent: rc = BBS_NONE
      uint32_t best = __reduce_min_sync(BB_FULL, cand);
      if (best == BBS_NONE && nR > ws.cbase) {   // the rest of G_ from memory, 128 per pass
        // sorted: G_ ascends in lead monomial (keys descend): a reducer whose key is below M's cannot divide, nor any after it
        const uint64_t stop = sorted ? M : 0ull;
        bool over = rlm[ws.cbase - 1] < stop;               // the last reducer of the register part
#pragma unroll 1
        for (int base = ws.cbase; base < nR && !over; base += 128) {
          const int r0 = base + lane, r1 = r0 + 32, r2 = r0 + 64, r3 = r0 + 96;
          const bool v0 = r0 < nR, v1 = r1 < nR, v2 = r2 < nR, v3 = r3 < nR;
          const uint64_t l0 = v0 ? rlm[r0] : ~0ull, l1 = v1 ? rlm[r1] : ~0ull, l2 = v2 ? rlm[r2] : ~0ull, l3 = v3 ? rlm[r3] : ~0ull;
          const bool h0 = v0 && ((mg - (l0 & K::ex_mask)) & K::ge_mask) == K::ge_mask, h1 = v1 && ((mg - (l1 & K::ex_mask)) & K::ge_mask) == K::ge_mask;
          const bool h2 = v2 && ((mg - (l2 & K::ex_mask)) & K::ge_mask) == K::ge_mask, h3 = v3 && ((mg - (l3 & K::ex_mask)) & K::ge_mask) == K::ge_mask;
          const uint32_t c2 = h0 ? (uint32_t)r0 : (h1 ? (uint32_t)r1 : (h2 ? (uint32_t)r2 : (h3 ? (uint32_t)r3 : BBS_NONE)));
          const uint32_t b2 = __reduce_min_sync(BB_FULL, c2);
          if (b2 != BBS_NONE) { best = (b2 << 16) | ridx[b2]; break; }
          over = __any_sync(BB_FULL, l0 < stop || l1 < stop || l2 < stop || l3 < stop);
        }
      }
      uint4 a = make_uint4(0u, 0u, 0u, 0u), b = make_uint4(0u, 0u, 0u, 0u), c = make_uint4((uint32_t)nR, 0u, 0u, 0u);
      if (best != BBS_NONE) {
        const GHead f = load_head(gh + (best & 0xffffu));
        const uint64_t adj = M - f.lm;            // key(LM h / LM f) - bias
        const uint64_t k = f.k1 + adj;
        const uint32_t sf = f.sug + (uint32_t)(f.lm >> K::dshift) - (uint32_t)(M >> K::dshift);   // >= 0: LM f divides M
        a = make_uint4((uint32_t)k, (uint32_t)(k >> 32), (uint32_t)adj, (uint32_t)(adj >> 32));
        b = make_uint4(f.invlc | (f.c1 << 16), f.off + 2u, f.off + f.len, 1u | ((f.len > 1u && (k & K::g_all)) ? 2u : 0u));
        c = make_uint4((best >> 16) + 1u, sf, 0u, 0u);
      }
      if (lane == 0) { sh.desc[half][0] = a; sh.desc[half][1] = b; sh.desc[half][2] = c; }
    }
  } else {
    // ---- stream warps: this thread's streams: its register slot, then its entries of the table
    uint64_t mk = ws.k0;
    uint32_t sc = 0u;        // this thread's part of M's coefficient: at most 1 + 768 / BBW_SLOTS values below 2^16
    if (mk == M) {
      sc = ws.c0;
      if (ws.p0 < ws.e0) {
        mk = ws.pk0 + ws.adj0;
        ws.c0 = bbf_mulmod(F, ws.pc0, ws.nc0);
        if (mk & K::g_all) ws.bad = 1u;
        ws.p0++;
        if (ws.p0 < ws.e0) { ws.pk0 = tk[ws.p0]; ws.pc0 = tc[ws.p0]; }   // the term behind the new head, needed a round later at the earliest
      } else {
        mk = ~0ull;
      }
      ws.k0 = mk;
    }
    if (ws.T > 0) {
#pragma unroll 1
      for (int i = tid; i < ws.T; i += BBW_SLOTS) {
        uint64_t k = st.key[i];
        if (k == M && k != ~0ull) {
          sc += st.coef[i];
          const uint32_t p = st.ptr[i];
          if (p < st.end[i]) {
            uint64_t kr; uint32_t cr;
            if (ws.pend_i == i) { kr = ws.pend_k; cr = ws.pend_c; ws.pend_i = -1; }
            else { kr = st.pkey[i]; cr = st.pcoef[i]; }
            k = kr + st.adj[i];
            const uint32_t c = bbf_mulmod(F, cr, st.nc[i]);
            if (k & K::g_all) ws.bad = 1u;
            st.key[i] = k; st.coef[i] = c; st.ptr[i] = p + 1u;
            if (p + 1u < st.end[i]) {
              if (ws.pend_i >= 0) { st.pkey[ws.pend_i] = ws.pend_k; st.pcoef[ws.pend_i] = ws.pend_c; }
              ws.pend_i = i; ws.pend_k = tk[p + 1u]; ws.pend_c = tc[p + 1u];
            }
          } else {
            k = ~0ull; st.key[i] = k;
          }
        }
        mk = k < mk ? k : mk;
      }
    }
    // the warp's first free register slot, the consumed monomial's coefficient sum, the 64-bit minimum through two 32-bit
    // reductions
    const uint32_t fm = __ballot_sync(BB_FULL, ws.k0 == ~0ull && tid < ws.regs);
    const uint32_t wsum = __reduce_add_sync(BB_FULL, sc);   // < 2^24
    const uint32_t hi = __reduce_min_sync(BB_FULL, (uint32_t)(mk >> 32));
    const uint32_t lo = __reduce_min_sync(BB_FULL, (uint32_t)(mk >> 32) == hi ? (uint32_t)mk : 0xffffffffu);
    const uint32_t fl = fm ? (uint32_t)(__ffs((int)fm) - 1) : BBW_NOFREE;
    if (lane == 0) sh.wrec[half][tid >> 5] = make_uint4(lo, hi, wsum | (fl << 24), 0u);
  }
#ifdef BBW_CLOCK
  const long long t1 = bbw_clock(0u);
  __syncthreads();
  ws.cw += t1 - t0;
#else
  __syncthreads();
#endif
  // every warp folds the stream warps' records, one per lane, and reads the descriptor
  {
    uint4 v = make_uint4(0xffffffffu, 0xffffffffu, BBW_NOFREE << 24, 0u);
    if (lane < BBW_WARPS - 1) v = sh.wrec[half][lane];
    dA = sh.desc[half][0]; dB = sh.desc[half][1]; dC = sh.desc[half][2];
    const uint32_t gs = __reduce_add_sync(BB_FULL, v.z & 0xffffffu);   // < 2^27
    const uint32_t hi = __reduce_min_sync(BB_FULL, v.y);
    const uint32_t lo = __reduce_min_sync(BB_FULL, v.y == hi ? v.x : 0xffffffffu);
    const uint32_t fr = __reduce_min_sync(BB_FULL, (v.z >> 24) != BBW_NOFREE ? ((uint32_t)lane << 5) | (v.z >> 24) : BBS_NONE);
    M2 = ((uint64_t)hi << 32) | lo; S = bbf_reduce(F, gs);
    freet = fr == BBS_NONE ? -1 : (int)fr;
  }
#ifdef BBW_CLOCK
  ws.tl = bbw_clock(S ^ (uint32_t)M2 ^ (uint32_t)freet ^ dA.x ^ dB.w ^ dC.x);   // behind the fold's results
  ws.cb += ws.tl - t1;
#endif
  half ^= 1;
}

// Opens a stream in register slot `target` (>= 0), else as the next entry of the table (the caller has checked the room):
// head key hk, the terms behind the head at [next, end), multiplier monomial adj; multiplier coefficient nc = -(S * invlc)
// and head coefficient c1 * nc are worked out by the one thread that owns the slot (icc = invlc | c1 << 16); S = 0 with
// icc = 1 | c << 16 opens a stream over a list as it is (multiplier 1).
__device__ __forceinline__ void wide_open(WideState& ws, WideStreams& st, const BBField F, int target, uint64_t hk, uint64_t adj,
                                          uint32_t S, uint32_t icc, uint32_t next, uint32_t end, const uint64_t* tk, const uint32_t* tc) {
  const int j = ws.T;
  int owner = target;
  if (target < 0) owner = j % BBW_SLOTS;
  if ((int)threadIdx.x == owner) {
    const uint32_t nc = S ? F.p - bbf_mulmod(F, S, icc & 0xffffu) : 1u;   // S * invlc != 0
    const uint32_t hc = bbf_mulmod(F, icc >> 16, nc);
    if (target >= 0) {
      ws.k0 = hk; ws.c0 = hc; ws.adj0 = adj; ws.nc0 = nc; ws.p0 = next; ws.e0 = end;
      if (next < end) { ws.pk0 = tk[next]; ws.pc0 = tc[next]; }
    } else {
      st.key[j] = hk; st.coef[j] = hc; st.adj[j] = adj; st.nc[j] = nc; st.ptr[j] = next; st.end[j] = end;
      if (next < end) {
        if (ws.pend_i >= 0) { st.pkey[ws.pend_i] = ws.pend_k; st.pcoef[ws.pend_i] = ws.pend_c; }
        ws.pend_i = j; ws.pend_k = tk[next]; ws.pend_c = tc[next];
      }
    }
  }
  if (target < 0) ws.T = j + 1;
#ifdef BBW_INSTR
  if (target < 0) ws.n_topen++;
#endif
}

// Consolidation (see the top of this file): h from its lead monomial M on goes to scratch half ws.cz in order, one stream over it
// (register slot 0) remains and M becomes its head monomial, all ones if nothing is left.  Returns the number of terms, -1
// if they do not fit `cap`.
template <int NV>
__device__ __forceinline__ int wide_consolidate(WideShared& sh, int& half, WideState& ws, WideStreams& st, const BBField F,
                                                uint64_t& M, uint64_t* tk, uint32_t* tc, uint32_t sbase, int cap) {
  const uint32_t base = sbase + (uint32_t)(ws.cz * cap);
  int t = 0;
  uint64_t m = M, fm = ~0ull; uint32_t fs = 0u;
#pragma unroll 1
  while (m != ~0ull) {
    uint64_t m2; uint32_t s; uint4 dA, dB, dC; int freet;
    wide_round<NV>(sh, half, ws, st, F, m, false, nullptr, nullptr, nullptr, 0, false, tk, tc, s, m2, dA, dB, dC, freet);
    if (s != 0u) {
      if (t >= cap) return -1;
      if (t == 0) { fm = m; fs = s; }
      if (threadIdx.x == 0) { tk[base + t] = m; tc[base + t] = s; }
      t++;
    }
    m = m2;
  }
  ws.pend_i = -1;   // every stream is exhausted: every slot is free
  ws.T = 0;
  ws.cz ^= 1;
  M = fm;
  __syncthreads();   // thread 0's list before thread 0 (the owner of slot 0) reads it back
  if (t > 0) wide_open(ws, st, F, 0, fm, 0ull, 0u, 1u | (fs << 16), base + 1u, base + (uint32_t)t, tk, tc);
  return t;
}

// reduce(spoly(G[i], G[j]), G_) (buchberger.cpp:18-49) by the block for the pair heads (hf, hg) and gamma = the key of the
// pair's lcm.  The remainder goes to (rk, rc) [cap rcap]; returns its length or a negative BB_STATUS_* on a fault; `steps`
// = reductions, `sug` = the sugar of the result (polynomials.cpp:150, 198).
template <int NV>
__device__ __forceinline__ int block_reduce_streams(const BBParams& P, const Env& e, WideShared& sh, int& half, WideState& ws,
                                                    WideStreams& st, const GHead hf, const GHead hg, const uint64_t gam, int& sug,
                                                    int& steps, uint64_t* rk, uint32_t* rc, int rcap, Ctr& ct) {
  typedef KL<NV> K;
  const BBField F = P.F;
  const GHeadMem* gh = ENV_PTR(GHeadMem, e, P, o_ghead);
  uint64_t* tk = ENV_PTR(uint64_t, e, P, o_tkey);
  uint32_t* tc = ENV_PTR(uint32_t, e, P, o_tcoef);
  const uint64_t* rlm = ENV_PTR(uint64_t, e, P, o_rlm);
  const uint32_t* ridx = ENV_PTR(uint32_t, e, P, o_ridx);
  const int nR = e.nG;
  const bool sorted = P.sort_reducers != 0;
  const int tid = threadIdx.x;
  int rlen = 0;
  steps = 0;
  ws.clear();
  if (tid >= BBW_SLOTS) {   // the control warp's part of G_ (G_ changes only between reductions)
#pragma unroll
    for (int q = 0; q < 8; q++) {
      const int r = (tid - BBW_SLOTS) + 32 * q;
      const bool in = r < nR && r < ws.cbase;
      ws.rl[q] = in ? (rlm[r] & K::ex_mask) : K::ex_mask;
      ws.rc[q] = in ? (((uint32_t)r << 16) | ridx[r]) : BBS_NONE;   // positions and basis indices are below 2^16
    }
  }
  // s = (gamma / LT f) tail(f) - (gamma / LT g) tail(g): the lead terms cancel exactly (buchberger.cpp:18-21); two streams
  // whose heads come from the head records, in register slots 0 and 1 (ws.regs >= 2)
  int opened = 0;
  if (hf.len > 1u) {
    const uint64_t adj = gam - hf.lm, k = hf.k1 + adj;
    if (k & K::g_all) return -BB_STATUS_OVERFLOW_EXPONENT;
    wide_open(ws, st, F, opened++, k, adj, F.p - 1u, hf.invlc | (hf.c1 << 16), hf.off + 2u, hf.off + hf.len, tk, tc);   // S = -1: nc = +invlc
  }
  if (hg.len > 1u) {
    const uint64_t adj = gam - hg.lm, k = hg.k1 + adj;
    if (k & K::g_all) return -BB_STATUS_OVERFLOW_EXPONENT;
    wide_open(ws, st, F, opened++, k, adj, 1u, hg.invlc | (hg.c1 << 16), hg.off + 2u, hg.off + hg.len, tk, tc);          // S = +1: nc = -invlc
  }
  // The block's threads agree on the lead monomial sequence, the streams and the faults; the reduction's bookkeeping
  // (remainder, counters, sugar) is left to ONE warp and published at the end: the last stream warp, whose slots fill last
  // (the control warp's round is the longest of the block, the first stream warps' come next).
  const int tbook = BBW_SLOTS - 32;
  const bool ctl = (tid >> 5) == BBW_WARPS - 2;
  int err = 0;
  uint32_t n_lms = 0u, n_tread = 0u;
  uint64_t M = ~0ull;   // pseudo lead monomial: consumes nothing, is no term of h
#pragma unroll 1
  do {
    uint64_t M2; uint32_t S; uint4 dA, dB, dC; int freet;
    wide_round<NV>(sh, half, ws, st, F, M, true, gh, rlm, ridx, nR, sorted, tk, tc, S, M2, dA, dB, dC, freet);
    if (M != ~0ull && S != 0u) {   // S == 0: the monomial cancelled, it is not a term of h
      if (ctl) {
        n_lms += dC.x;
        if (dB.w & 1u) {
          const int sf = (int)dC.y;
          sug = sf > sug ? sf : sug;
          n_tread += dB.z - dB.y + 2u;   // |f|
          steps++;
        } else {          // no divisor: the lead term moves to the remainder (beyond its capacity: counted, not written)
          if (rlen < rcap && tid == tbook) { rk[rlen] = M; rc[rlen] = S; }
          rlen++;
        }
      }
      if ((dB.w & 1u) && dB.z + 1u > dB.y) {   // h <- h - (LT h / LT f) f, |f| > 1: the lead terms cancel, f's tail becomes a stream
        if (dB.w & 2u) { err = -BB_STATUS_OVERFLOW_EXPONENT; break; }
        if (freet < 0 && ws.T >= ws.tcap) {   // no register slot, no room in the table
#ifdef BBW_INSTR
          ws.n_consol++;
#endif
          const int t = wide_consolidate<NV>(sh, half, ws, st, F, M2, tk, tc, (uint32_t)P.max_terms, P.max_poly_terms);
          if (t < 0) { err = -BB_STATUS_OVERFLOW_SCRATCH; break; }
          freet = t > 0 ? 1 : 0;
        }
        const uint64_t k = ((uint64_t)dA.y << 32) | dA.x;
        wide_open(ws, st, F, freet, k, ((uint64_t)dA.w << 32) | dA.z, S, dB.x, dB.y, dB.z, tk, tc);
        M2 = k < M2 ? k : M2;
      }
    }
    M = M2;
#ifdef BBW_CLOCK
    { const long long t3 = bbw_clock((uint32_t)M ^ ws.c0 ^ (uint32_t)ws.k0); ws.cp += t3 - ws.tl; ws.tl = t3; }
#endif
  } while (M != ~0ull);
  if (tid == tbook) {
    sh.fin[0] = make_uint4((uint32_t)(err ? err : (rlen > rcap ? -BB_STATUS_OVERFLOW_TERMS : rlen)), (uint32_t)steps, (uint32_t)sug, 0u);
    sh.fin[1] = make_uint4(n_lms, n_tread, (uint32_t)(rlen < rcap ? rlen : rcap), 0u);
  }
  const int bad = __syncthreads_or(ws.bad != 0u);   // also: the book-keeping warp's remainder and counts before the others read them
  const uint4 f0 = sh.fin[0], f1 = sh.fin[1];
  steps = (int)f0.y; sug = (int)f0.z;
  ct.lms += f1.x; ct.tread += f1.y; ct.moves += f1.z;
  if ((int)f0.x < 0) return (int)f0.x;
  if (bad) return -BB_STATUS_OVERFLOW_EXPONENT;
  return (int)f0.x;
}

// Removes row `row` from the pair list keeping order (buchberger.cpp:319), by the whole block: chunk by chunk, read, barrier,
// write one place lower.  The pair and its cached lcm key go to (pr, gam).  e.nP is NOT changed here.
__device__ __forceinline__ void block_take_pair(const BBParams& P, const Env& e, int row, uint32_t& pr, uint64_t& gam) {
  uint32_t* pairs = ENV_PTR(uint32_t, e, P, o_pairs);
  uint64_t* plcm = ENV_PTR(uint64_t, e, P, o_plcm);
  pr = pairs[row];
  gam = plcm[row];
#pragma unroll 1
  for (int b0 = row; b0 < e.nP - 1; b0 += BBW_THREADS) {
    const int idx = b0 + threadIdx.x;
    const bool v = idx < e.nP - 1;
    uint32_t x = 0u; uint64_t y = 0ull;
    if (v) { x = pairs[idx + 1]; y = plcm[idx + 1]; }
    __syncthreads();   // every read of this chunk (and of (pr, gam) in the first) before any write
    if (v) { pairs[idx] = x; plcm[idx] = y; }
  }
}

// update() (buchberger.cpp:52-99) + reducer-list insertion by the BLOCK for Gebauer-Moeller elimination and more than 64
// basis elements; result as warp_add_basis (bb_device.cuh), to every thread.  On cyclic-6 the basis has ~600 (up to ~1200)
// elements when one is added, and warp_add_basis's peeling loop -- one sweep of all L_i = lcm(LM_i, LM f) per kept lcm, ~16
// of them -- took 66 K cycles per update with seven warps waiting: 7 % of an episode (clock probes, profiles/README.md).
// Here warp 0 prepares (the L_i into the slot's scratch array, the old-pair filter, :63-70), the sweep of a kept lcm is
// split over the warps (warp w takes chunks w, w + BBW_WARPS, ...; one barrier and one fold of BBW_WARPS records per kept
// lcm; the thread that reads an entry is the one that writes it), and warp 0 finishes (new pairs in ascending i, reducer
// list, head record).  Statement for statement the general path of warp_add_basis otherwise; everything else goes there.
template <int NV>
__device__ __forceinline__ long long block_add_basis(const BBParams& P, WideShared& sh, unsigned char* base, int m, int nP,
                                                     int off, int len, int sug) {
  typedef KL<NV> K;
  const auto& H = BB_HOT(P);
  const int tid = threadIdx.x, lane = bb_lane(), warp = tid >> 5;
  if (H.elimination != BB_ELIM_GEBAUERMOELLER || m <= 64 || m >= H.max_basis) {
    if (tid < 32) {
      const long long r = warp_add_basis<NV>(P, base, m, nP, off, len, sug);
      if (tid == 0) sh.upd = r;
    }
    __syncthreads();
    return sh.upd;
  }
  const uint32_t ltm = bb_lt_mask();
  base = bb_global(base);
  const uint64_t* tk = reinterpret_cast<const uint64_t*>(base + H.o_tkey) + off;
  const uint32_t* tc = reinterpret_cast<const uint32_t*>(base + H.o_tcoef) + off;
  const uint64_t fk = tk[0];
  uint64_t* lm = reinterpret_cast<uint64_t*>(base + H.o_lm);
  uint64_t* lscr = reinterpret_cast<uint64_t*>(base + H.o_lscr);
  uint64_t* plcm = reinterpret_cast<uint64_t*>(base + H.o_plcm);
  uint32_t* pairs = reinterpret_cast<uint32_t*>(base + H.o_pairs);
  // ---- every thread: lscr[i] = key of L_i (the old-pair filter gathers from it)
  bool ovf = false;  // deg(L_i) must fit the degree field: bit 63 is a tag below, never a silently wrapped degree
#pragma unroll 1
  for (int i = tid; i < m; i += BBW_THREADS) {
    const uint64_t le = K::lcm_exps(lm[i], fk);
    const uint32_t dg = K::sum_fields(le);
    ovf |= dg > K::dmax;
    lscr[i] = le | ((uint64_t)(K::dmax - dg) << K::dshift);
  }
  if (__syncthreads_or(ovf)) return -3;
  // ---- warp 0: (1) old pairs (i, j) dropped iff LM f | lcm_ij and lcm_ij != L_i and lcm_ij != L_j (:63-70)
  if (tid < 32) {
    const uint64_t fe = fk & K::ex_mask;
    int w = 0;
#pragma unroll 1
    for (int b0 = 0; b0 < nP; b0 += 32) {
      const int idx = b0 + lane;
      const bool valid = idx < nP;
      uint32_t pr = 0u; uint64_t pl = 0ull;
      bool keep = false;
      if (valid) {
        pr = pairs[idx]; pl = plcm[idx];
        const uint64_t l = pl & K::ex_mask;
        const bool drop = K::divides(fe, l) && l != (lscr[pr & 0xffffu] & K::ex_mask) && l != (lscr[pr >> 16] & K::ex_mask);
        keep = !drop;
      }
      const uint32_t km = __ballot_sync(BB_FULL, keep);
      if (keep) {  // w + rank <= idx: never overtakes an unread entry of a later chunk
        const int pos = w + __popc(km & ltm);
        pairs[pos] = pr; plcm[pos] = pl;
      }
      w += __popc(km);
      __syncwarp();
    }
    if (tid == 0) sh.upd = w;
  }
  __syncthreads();   // the filter reads the keys the sweeps below start to overwrite
  // ---- every thread: (2)-(4) by peeling.  The smallest remaining L (largest key; lowest index among equals) cannot be
  // strictly divided by anything still alive; it kills every multiple (strict or equal), and its pair is emitted unless a
  // member of its group is coprime to f.  lscr[i] = key while undecided, 0 once dead, key | 1 << 63 once chosen.  Entry i
  // belongs to the thread that sweeps it: lane i % 32 of warp (i / 32) % BBW_WARPS.
  uint64_t kk = 0ull, kkey = 0ull;   // exponents / key of the current kept lcm
  int kidx = -1, buf = 0;
  for (;;) {
    uint64_t bk = 0ull; int bi = 0x7fffffff;
    uint32_t cop_any = 0u;
#pragma unroll 1
    for (int b0 = warp * 32; b0 < m; b0 += BBW_THREADS) {
      const int i = b0 + lane;
      uint64_t x = i < m ? lscr[i] : 0ull;
      bool und = x != 0ull && (long long)x > 0;  // undecided
      if (kidx >= 0) {
        const uint64_t ei = x & K::ex_mask;
        const bool eq = x != 0ull && ei == kk;    // the kept lcm itself included
        if (und && ((((ei | K::ge_mask) - kk) & K::ge_mask) == K::ge_mask)) { lscr[i] = 0ull; und = false; }
        bool cop = false;
        if (eq) cop = K::coprime(lm[i], fk);
        cop_any |= __ballot_sync(BB_FULL, cop);
      }
      if (und && x > bk) { bk = x; bi = i; }  // ascending i per lane: first occurrence kept on ties
    }
    {   // the warp's largest undecided key, lowest index among equals
      const uint32_t hi = __reduce_max_sync(BB_FULL, (uint32_t)(bk >> 32));
      const bool c1 = (uint32_t)(bk >> 32) == hi;
      const uint32_t lo = __reduce_max_sync(BB_FULL, c1 ? (uint32_t)bk : 0u);
      const bool c2 = c1 && (uint32_t)bk == lo;
      const uint32_t wi = __reduce_min_sync(BB_FULL, c2 ? (uint32_t)bi : 0x7fffffffu);
      if (lane == 0) sh.prec[buf][warp] = make_uint4(lo, hi, wi, cop_any ? 1u : 0u);
    }
    __syncthreads();
    uint4 v = make_uint4(0u, 0u, 0x7fffffffu, 0u);
    if (lane < BBW_WARPS) v = sh.prec[buf][lane];
    buf ^= 1;
    const bool grp_cop = __any_sync(BB_FULL, v.w != 0u);
    const uint32_t hi = __reduce_max_sync(BB_FULL, v.y);
    const uint32_t lo = __reduce_max_sync(BB_FULL, v.y == hi ? v.x : 0u);
    const uint32_t ni = __reduce_min_sync(BB_FULL, (v.y == hi && v.x == lo) ? v.z : 0x7fffffffu);
    // the kept lcm whose sweep this was: chosen for emission unless its group has a coprime member (by the entry's owner)
    if (kidx >= 0 && ((kidx >> 5) & (BBW_WARPS - 1)) == warp && (kidx & 31) == lane) lscr[kidx] = grp_cop ? 0ull : (kkey | (1ull << 63));
    if ((hi | lo) == 0u) break;   // nothing undecided
    kidx = (int)ni;
    kkey = ((uint64_t)hi << 32) | lo;
    kk = kkey & K::ex_mask;
    // decided: out of the undecided set while it sweeps (by the entry's owner, the only thread that reads it in a sweep)
    if (((kidx >> 5) & (BBW_WARPS - 1)) == warp && (kidx & 31) == lane) lscr[kidx] = kkey | (1ull << 63);
  }
  __syncthreads();   // every owner's marks before warp 0 reads them
  nP = (int)sh.upd;
  // ---- warp 0: (5) new pairs in ascending i (:86) behind the survivors (:91-92), the reducer list, the head record
  if (tid < 32) {
    long long r = 0;
    int emitted = 0;
#pragma unroll 1
    for (int b0 = 0; b0 < m && r == 0; b0 += 32) {
      const int i = b0 + lane;
      const uint64_t x = i < m ? lscr[i] : 0ull;
      const bool keep = (long long)x < 0;
      const uint32_t km = __ballot_sync(BB_FULL, keep);
      const int cnt = __popc(km);
      if (nP + cnt > H.max_pairs) { r = -1; break; }
      if (keep) {
        const int pos = nP + __popc(km & ltm);
        pairs[pos] = ((uint32_t)m << 16) | (uint32_t)i;
        plcm[pos] = x & ~(1ull << 63);
      }
      nP += cnt; emitted += cnt;
    }
    if (r == 0) {
      // upper_bound by lead monomial when sort_reducers (buchberger.cpp:308-311 / 323-326), else appended
      uint64_t* rlm = reinterpret_cast<uint64_t*>(base + H.o_rlm);
      uint32_t* ridx = reinterpret_cast<uint32_t*>(base + H.o_ridx);
      int pos = m;
      if (H.sort_reducers) {
        int cnt = 0;  // reducers with LM <= new LM  <=>  key >= new key
#pragma unroll 1
        for (int b0 = 0; b0 < m; b0 += 32) {
          const int q = b0 + lane;
          cnt += __popc(__ballot_sync(BB_FULL, q < m && rlm[q] >= fk));
        }
        pos = cnt;
#pragma unroll 1
        for (int hi = m; hi > pos; hi -= 32) {
          const int lo = hi - 32 > pos ? hi - 32 : pos;
          const int idx = lo + lane;
          const bool in = idx < hi;
          uint64_t k = 0; uint32_t ix = 0;
          if (in) { k = rlm[idx]; ix = ridx[idx]; }
          __syncwarp();
          if (in) { rlm[idx + 1] = k; ridx[idx + 1] = ix; }
          __syncwarp();
        }
      }
      if (lane == 0) {
        rlm[pos] = fk; ridx[pos] = (uint32_t)m;
        lm[m] = fk;
        GHeadMem* g = reinterpret_cast<GHeadMem*>(base + H.o_ghead) + m;
        const uint32_t inv = bb_global(H.invtab)[tc[0]];
        const uint64_t k1 = len > 1 ? tk[1] : 0ull;
        const uint32_t c1 = len > 1 ? tc[1] : 0u;
        reinterpret_cast<uint4*>(g)[0] = make_uint4((uint32_t)fk, (uint32_t)(fk >> 32), (uint32_t)k1, (uint32_t)(k1 >> 32));
        reinterpret_cast<uint4*>(g)[1] = make_uint4(inv | (c1 << 16), (uint32_t)sug, (uint32_t)off, (uint32_t)len);
      }
      __syncwarp();
      r = ((long long)emitted << 32) | (long long)nP;
    }
    if (tid == 0) sh.upd = r;
  }
  __syncthreads();
  return sh.upd;
}

// One environment step by the whole CTA (BuchbergerEnv::step, buchberger.cpp:318-329, with the pair chosen by
// `strategy`).  e and every scalar below are block-uniform.  Pair selection and update() (Gebauer-Moeller) are the warp
// routines of bb_device.cuh run by warp 0.  Returns the number of polynomial additions; `pair` receives (j << 16) | i.
template <int NV>
__device__ __forceinline__ int block_step(const BBParams& P, Env& e, WideShared& sh, int& half, WideState& ws, WideStreams& st,
                                          int strategy, uint32_t* sel_rng, uint32_t& pair, Ctr& ct) {
  typedef KL<NV> K;
  const int tid = threadIdx.x;
#ifdef BBW_CLOCK
  const long long c0 = bbw_clock(0u);
#endif
  if (tid < 32) {   // warp 0: select the pair
    const int row = warp_select<NV>(P, e, strategy, sel_rng);
    if (tid == 0) sh.row = row;
  }
  __syncthreads();
#ifdef BBW_CLOCK
  const long long c1 = bbw_clock((uint32_t)sh.row);
#endif
  uint32_t pr; uint64_t gam;
  block_take_pair(P, e, sh.row, pr, gam);
  e.nP--;
  pair = pr;
#ifdef BBW_CLOCK
  const long long c2 = bbw_clock(pr ^ (uint32_t)gam);
  ws.s_sel += c1 - c0; ws.s_take += c2 - c1;
#endif
  const GHeadMem* gh = ENV_PTR(GHeadMem, e, P, o_ghead);
  const GHead hf = load_head(gh + (pr & 0xffffu)), hg = load_head(gh + (pr >> 16));
  e.guard |= gam;
  ct.tread += hf.len + hg.len;
  int sug;
  {  // sugar of the S-polynomial: max(deg(gamma / LM f) + sug f, deg(gamma / LM g) + sug g)
    const int cg0 = (int)(uint32_t)(gam >> K::dshift);
    const int sf = (int)hf.sug + (int)(uint32_t)(hf.lm >> K::dshift) - cg0, sg = (int)hg.sug + (int)(uint32_t)(hg.lm >> K::dshift) - cg0;
    sug = sf > sg ? sf : sg;
  }
  if (e.guard & K::g_all) { e.status = BB_STATUS_OVERFLOW_EXPONENT; return 1; }
  int steps = 0;
  const int rlen = block_reduce_streams<NV>(P, e, sh, half, ws, st, hf, hg, gam, sug, steps, ENV_PTR(uint64_t, e, P, o_tkey) + e.nT,
                                            ENV_PTR(uint32_t, e, P, o_tcoef) + e.nT, P.max_terms - e.nT, ct);
#ifdef BBW_CLOCK
  const long long c3 = bbw_clock((uint32_t)rlen);
  ws.s_red += c3 - c2;
#endif
  if (rlen < 0) { e.status = -rlen; return 1 + steps; }
  if (rlen > 0) {
    ct.upb += (unsigned)e.nG; ct.upp += (unsigned)e.nP;
    const long long r = block_add_basis<NV>(P, sh, e.base, e.nG, e.nP, e.nT, rlen, sug);
    if (r < 0) {
      e.status = (r == -1) ? BB_STATUS_OVERFLOW_PAIRS : (r == -2 ? BB_STATUS_OVERFLOW_BASIS : BB_STATUS_OVERFLOW_EXPONENT);
      return 1 + steps;
    }
    e.nP = (int)(r & 0xffffffffll);
    ct.upp += (unsigned)(r >> 32);
    e.nG++; e.nT += rlen;
#ifdef BBW_CLOCK
    ws.s_upd += bbw_clock((uint32_t)e.nP) - c3;
#endif
  }
  if (e.nP == 0) e.status = BB_STATUS_DONE;
  return 1 + steps;
}
