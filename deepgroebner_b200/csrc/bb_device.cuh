// bb_device.cuh -- warp-per-environment Buchberger step for sm_100a (v2: compact hot loop).
//
// One warp owns one environment slot.  All scalars of the slot (|G|, |P|, arena cursor, the dividend's first two
// terms, ...) are warp-uniform register values; all per-slot arrays live in ONE contiguous arena per slot in HBM
// (L1/L2 resident in practice) and are accessed lane-strided, i.e. coalesced.  No block-level synchronisation on
// the step path.
//
// What v1's profile (profiles/r01_v1_*) showed and what this file does about it:
//   * 52 % of stall samples were instruction fetch (10.7 K SASS instructions, every helper inlined 2-3 times)
//     -> the layout is a compile-time template parameter (KL<NV>), cold paths (reset + generator, final GB, hashes,
//        the general merge) are __noinline__ single copies that talk to the caller through the slot's state record,
//        and the hot loop is select -> erase -> spoly -> reduce -> add_basis only.
//   * 1743 warp instructions per env-step -> polynomials with <= 2 terms (every polynomial of a binomial ideal)
//     never touch the merge: the dividend's first two terms live in registers, each basis element has a 32-byte
//     head record (lead monomial, 1/LC, second term) fetched with two 128-bit loads, and every pair caches the
//     key of its lcm so selection and the Gebauer-Moeller sweep read one coalesced array.
//   * 124 registers -> counters are 7 x u32 spilled to shared memory per episode, slot pointers are one base.
//
// Reference semantics followed (deepgroebner/buchberger.cpp, polynomials.cpp) are cited at each function.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/bbenv.h"
#include "bb_layout.cuh"

#define BB_FULL 0xffffffffu
#ifndef BB_ADD_BASIS_INLINE
#define BB_ADD_BASIS_INLINE __noinline__   // A/B switch: __forceinline__ puts update() into every caller
#endif
#define BB_GOLD 0x9E3779B97F4A7C15ULL
#define BB_GOLD2 0xD1B54A32D192ED03ULL

// ---------------------------------------------------------------------------------------------------- parameters
struct __align__(16) BBEnvState {  // one per slot, 96 bytes
  int nG, nP, nT, status;
  int steps, adds, zero, nonzero;
  int rerolls, episode, truncated;
  unsigned sel_rng;              // minstd_rand0 state of Random selection (buchberger.cpp:190-197)
  unsigned long long trace_hash;
  unsigned long long rng;        // minstd_rand0 state of this environment's ideal stream
  double disc_return, discount;
  unsigned long long pad2[2];
};

// Head record of a basis element: everything a 2-term polynomial needs, and the arena range of the full term list.
// Head record of a basis element as it sits in the arena (32 bytes, two 128-bit loads) ...
struct __align__(32) GHeadMem {
  uint64_t lm;     // lead monomial key
  uint64_t k1;     // second term's key (undefined when len == 1)
  uint32_t ic;     // (1 / lead coefficient) | (second term's coefficient << 16): both are < p < 2^16
  uint32_t sug;    // sugar degree (Polynomial::sug, polynomials.h:93)
  uint32_t off;    // first term's index in the slot's term arena
  uint32_t len;    // number of terms
};
// ... and unpacked in (warp-uniform) registers
struct GHead {
  uint64_t lm, k1;
  uint32_t invlc, c1, sug, off, len;
};

struct BBDist {           // RandomBinomialIdealGenerator / RandomIdealGenerator parameters (ideals.cpp:157-231)
  int enabled, d, s, homogeneous, pure, ncp;
  int kind;               // 0: binomials (ideals.cpp:168-201); 1: Poisson-length polynomials (ideals.cpp:214-231)
  double lm_thr;          // kind 1: exp(-lam), std::poisson_distribution::param_type::_M_lm_thr for mean < 12
  const double* cp;       // [d+1] cumulative degree probabilities (libstdc++ discrete_distribution::_M_cp)
  const uint64_t* basis;  // packed monomials of degree 0..d, lex-descending within a degree (ideals.cpp:39-64)
  const int* basis_off;   // [d+2]
};

struct BBPre;   // prefetch queues of the step API (bb_kernels.cuh)

struct BBParams {
  BBField F;
  int nvars;
  int num_envs, k, cols, elimination, rewards, sort_input, sort_reducers;
  int max_basis, max_pairs, max_terms, max_poly_terms, max_gens, max_gen_terms;
  // one contiguous arena per slot: base = arena + slot * slot_stride; byte offsets of the arrays inside it
  unsigned char* arena;
  unsigned long long slot_stride;
  unsigned o_ghead;   // GHeadMem[max_basis]          by basis index
  unsigned o_lm;      // u64     [max_basis]          lead monomial key by basis index
  unsigned o_rlm;     // u64     [max_basis]          reducer list G_ in scan order: lead monomial key
  unsigned o_lscr;    // u64     [max_basis]          update() scratch: lcm(LM_i, LM f) exponents | coprime << 63
  unsigned o_plcm;    // u64     [max_pairs]          key of lcm(LM_i, LM_j) of each pair, in P order
  unsigned o_tkey;    // u64     [max_terms]          term arena: packed monomials
  unsigned o_hkey;    // u64     [2][max_poly_terms]  dividend ping-pong scratch
  unsigned o_ridx;    // u32     [max_basis]          reducer list: basis index
  unsigned o_pairs;   // u32     [max_pairs]          pair list P in order: (j << 16) | i
  unsigned o_tcoef;   // u32     [max_terms]          term arena: coefficients
  unsigned o_hcoef;   // u32     [2][max_poly_terms]
  unsigned o_logit;   // f32     [max_pairs]          policy head scratch: one logit per pair row
  int auto_reset;     // k_step / k_rollout: a finished environment is reset in the same call (vector-env semantics)
  int max_episode_length;  // k_step / k_rollout: 0 = unlimited; else an episode is cut (BB_STATUS_TRUNCATED, done = 1) once it
                           // has MORE than this many steps -- `episode_length > max_episode_length: break`, pg.py:470-471
  int obs_nv;         // variables shown per monomial in the state matrix (= nvars; less only under bb_set_obs_nvars)
  BBEnvState* st;
  // staged input ideals, one per slot
  uint64_t* in_key; uint32_t* in_coef;  // [num_envs][max_gen_terms], each polynomial sorted descending
  int* in_off;                          // [num_envs][max_gens+1]; in_off[0] = 0, in_off[npoly] = nterms
  int* in_np;                           // [num_envs]
  // reduced-GB output arena, one per slot
  uint64_t* gkey; uint32_t* gcoef;      // [num_envs][max_terms]
  int* glen;                            // [num_envs][max_basis]
  int* gcount;                          // [num_envs][2] = (npolys, nterms)
  uint64_t* grlm; uint32_t* gridx; uint32_t* gflag;  // [num_envs][max_basis] scratch of warp_final_gb
  BBDist dist;
  const BBPre* pre;                     // per-environment queues of prepared next episodes (NULL: none), see warp_next_episode
  const uint16_t* invtab;               // [p] multiplicative inverses in GF(p) (invtab[0] = 0)
  unsigned long long* counters;         // bb_counters as 12 x u64
};

enum { CT_STEPS = 0, CT_ADDS, CT_TREAD, CT_TWRITE, CT_LMS, CT_MOVES, CT_UPB, CT_UPP, CT_OBS, CT_NONZERO, CT_ZERO,
       CT_EPISODES, CT_COUNT };

// Per-warp traffic counters of the step path (warp-uniform u32 registers; spilled to the warp's u64 row in shared
// memory at least once per episode, so they cannot wrap).  Step / addition / episode counts are added to the row by
// the kernels directly.
struct Ctr {
  uint32_t tread, twrite, lms, moves, upb, upp, obs;
  __device__ __forceinline__ void clear() { tread = twrite = lms = moves = upb = upp = obs = 0; }
  __device__ __forceinline__ void spill(unsigned long long* row) {  // row: this warp's CT_COUNT accumulators
    if ((threadIdx.x & 31) == 0) {
      row[CT_TREAD] += tread; row[CT_TWRITE] += twrite; row[CT_LMS] += lms; row[CT_MOVES] += moves;
      row[CT_UPB] += upb; row[CT_UPP] += upp; row[CT_OBS] += obs;
    }
    clear();
  }
};

// Warp-uniform view of one slot.
struct Env {
  unsigned char* base;
  int nG, nP, nT, status;
  uint64_t guard;  // OR of every produced monomial key: any guard bit set => exponent/degree overflow
};

// Every arena lives in global memory: saying so lets the compiler emit LDG / STG instead of generic LD / ST (whose
// address-space resolution sits on the latency chain of every dependent load of the step).
template <class T>
__device__ __forceinline__ T* bb_global(T* p) {
  __builtin_assume(__isGlobal(p));
  return p;
}
#define ENV_PTR(T, e, P, off) (bb_global(reinterpret_cast<T*>((e).base + (P).off)))
#define SLOT_PTR(T, P, slot, off) (bb_global(reinterpret_cast<T*>((P).arena + (size_t)(slot) * (P).slot_stride + (P).off)))

__device__ __forceinline__ int bb_lane() { return threadIdx.x & 31; }
__device__ __forceinline__ uint32_t bb_lt_mask() { return (1u << bb_lane()) - 1u; }
__device__ __forceinline__ uint64_t bb_shfl64(uint64_t v, int src) {
  uint32_t lo = __shfl_sync(BB_FULL, (uint32_t)v, src);
  uint32_t hi = __shfl_sync(BB_FULL, (uint32_t)(v >> 32), src);
  return ((uint64_t)hi << 32) | lo;
}
__device__ __forceinline__ uint64_t bb_mix64(uint64_t z) {
  z ^= z >> 30; z *= 0xbf58476d1ce4e5b9ULL;
  z ^= z >> 27; z *= 0x94d049bb133111ebULL;
  z ^= z >> 31;
  return z;
}
__host__ __device__ __forceinline__ uint64_t bb_hash_item_impl(uint64_t x, uint64_t pos) {
  uint64_t z = x + BB_GOLD * (pos + 1);
  z ^= z >> 30; z *= 0xbf58476d1ce4e5b9ULL;
  z ^= z >> 27; z *= 0x94d049bb133111ebULL;
  z ^= z >> 31;
  return z;
}

__device__ __forceinline__ void env_load(const BBParams& P, int slot, Env& e) {
  e.base = bb_global(P.arena + (size_t)slot * P.slot_stride);
  const int4 s = *reinterpret_cast<const int4*>(bb_global(&P.st[slot]));
  e.nG = s.x; e.nP = s.y; e.nT = s.z; e.status = s.w;
  e.guard = 0;
}
__device__ __forceinline__ void env_store(const BBParams& P, int slot, const Env& e) {
  if (bb_lane() == 0) *reinterpret_cast<int4*>(&P.st[slot]) = make_int4(e.nG, e.nP, e.nT, e.status);
}
__device__ __forceinline__ GHead load_head(const GHeadMem* g) {
  const uint4 a = reinterpret_cast<const uint4*>(g)[0], b = reinterpret_cast<const uint4*>(g)[1];
  GHead h;
  h.lm = ((uint64_t)a.y << 32) | a.x; h.k1 = ((uint64_t)a.w << 32) | a.z;
  h.invlc = b.x & 0xffffu; h.c1 = b.x >> 16; h.sug = b.y; h.off = b.z; h.len = b.w;
  return h;
}

// ---------------------------------------------------------------------------------------------------- random streams
// minstd_rand0 + libstdc++ distributions restated (ideals.h:177-179; SURVEY Appendix B): the streams must match
// the reference generator bit for bit because "identical seeded inputs" is part of the parity contract.
// The engine state is < 2^31, so everything is 32-bit arithmetic except the 46-bit product.
__device__ __forceinline__ uint32_t rng_seed(int seed) {
  unsigned long long s = (unsigned long long)(long long)seed % 2147483647ULL;  // int -> unsigned long, then mod m
  return s == 0 ? 1u : (uint32_t)s;
}
__device__ __forceinline__ uint32_t rng_next(uint32_t& x) {
  const unsigned long long pr = (unsigned long long)x * 16807ULL;       // < 2^46
  uint32_t r = (uint32_t)(pr & 0x7fffffffULL) + (uint32_t)(pr >> 31);  // 2^31 == 1 (mod 2^31 - 1)
  if (r >= 2147483647u) r -= 2147483647u;
  x = r;
  return r;
}
// uniform_int_distribution<int>(a,b): "fallback (2 divisions)" branch of bits/uniform_int_dist.h
__device__ __forceinline__ int rng_uniform(uint32_t& x, int a, int b) {
  const uint32_t urngrange = 2147483645u;
  const uint32_t uerange = (uint32_t)(b - a) + 1u;
  const uint32_t scaling = urngrange / uerange, past = uerange * scaling;
  uint32_t ret;
  do ret = rng_next(x) - 1u; while (ret >= past);
  return a + (int)(ret / scaling);
}
// generate_canonical<double,53>: two draws, (u1-1) + (u2-1)*R over R*R, all in round-to-nearest double ops
__device__ __forceinline__ double rng_canonical(uint32_t& x) {
  const double R = 2147483646.0;
  double s = (double)(rng_next(x) - 1u);
  s = __dadd_rn(s, __dmul_rn((double)(rng_next(x) - 1u), R));
  double r = __ddiv_rn(s, __dmul_rn(R, R));
  if (r >= 1.0) r = __longlong_as_double(0x3FEFFFFFFFFFFFFFLL);  // nextafter(1,0)
  return r;
}
__device__ __forceinline__ int rng_degree(const BBDist& D, uint32_t& x) {
  if (D.ncp < 2) return 0;
  const double p = rng_canonical(x);
  int lo = 0, hi = D.ncp;
  while (lo < hi) { int mid = (lo + hi) >> 1; if (D.cp[mid] < p) lo = mid + 1; else hi = mid; }
  return lo;
}

// ---------------------------------------------------------------------------------------------------- merge
// out = cA * mA * A  +  cB * mB * B     (Polynomial operator+ / Term*Polynomial, polynomials.cpp:148-202)
// A, B: term lists in ascending key order (descending grevlex), coefficients in [1,p).  adjX = key(mX) - bias.
// Cancelled terms are dropped.  Warp-cooperative merge path: every round each lane holds one element of each
// 32-wide window, finds its merged rank by a shuffle binary search in the other window, equal monomials are
// paired (A carries the sum, B retires), and the survivors are scattered in rank order.
// Returns the number of output terms, -1 if `cap` would be exceeded, -3 if a produced key has a guard bit set.
// One out-of-line copy: polynomials with more than two terms are the only callers.
template <int NV>
__device__ __noinline__ int warp_merge(BBField F, const uint64_t* __restrict__ Ak, const uint32_t* __restrict__ Ac, int nA,
                                       uint32_t cA, uint64_t adjA, const uint64_t* __restrict__ Bk,
                                       const uint32_t* __restrict__ Bc, int nB, uint32_t cB, uint64_t adjB,
                                       uint64_t* __restrict__ Ok, uint32_t* __restrict__ Oc, int cap) {
  typedef KL<NV> K;
  const int lane = bb_lane();
  int ia = 0, ib = 0, no = 0;
  uint64_t guard = 0;
  if (nB == 0 || nA == 0) {  // scaled copy
    const uint64_t* Sk = nB == 0 ? Ak : Bk; const uint32_t* Sc = nB == 0 ? Ac : Bc;
    const int nS = nB == 0 ? nA : nB; const uint32_t cS = nB == 0 ? cA : cB; const uint64_t adjS = nB == 0 ? adjA : adjB;
    if (nS > cap) return -1;
#pragma unroll 1
    for (int t = lane; t < nS; t += 32) {
      uint64_t k = Sk[t] + adjS; guard |= k;
      Ok[t] = k; Oc[t] = (cS == 1u) ? Sc[t] : bbf_mulmod(F, Sc[t], cS);
    }
    return __any_sync(BB_FULL, (guard & K::g_all) != 0ull) ? -3 : nS;
  }
  while (ia < nA || ib < nB) {
    uint64_t ak = ~0ull, bk = ~0ull;
    uint32_t ac = 0, bc = 0;
    const bool va = ia + lane < nA, vb = ib + lane < nB;
    if (va) { ak = Ak[ia + lane] + adjA; guard |= ak; ac = (cA == 1u) ? Ac[ia + lane] : bbf_mulmod(F, Ac[ia + lane], cA); }
    if (vb) { bk = Bk[ib + lane] + adjB; guard |= bk; bc = (cB == 1u) ? Bc[ib + lane] : bbf_mulmod(F, Bc[ib + lane], cB); }
    // rank of my A element: lane + #{b < a};  of my B element: lane + #{a <= b}  (A first on ties)
    int ca = 0, cb = 0;
#pragma unroll
    for (int step = 16; step; step >>= 1) {
      uint64_t vB = bb_shfl64(bk, ca + step - 1);
      uint64_t vA = bb_shfl64(ak, cb + step - 1);
      if (vB < ak) ca += step;
      if (vA <= bk) cb += step;
    }
    {
      uint64_t vB = bb_shfl64(bk, ca), vA = bb_shfl64(ak, cb);
      if (vB < ak) ca++;
      if (vA <= bk) cb++;
    }
    // partners: first b >= a sits at index ca; last a <= b sits at index cb-1
    uint64_t pB = bb_shfl64(bk, ca & 31);
    uint32_t pBc = __shfl_sync(BB_FULL, bc, ca & 31);
    uint64_t pA = bb_shfl64(ak, (cb - 1) & 31);
    const bool partA = va && ca < 32 && pB == ak;
    const bool partB = vb && cb > 0 && pA == bk;
    const int ra = lane + ca, rb = lane + cb;
    const bool emitA = va && ra < 32 && !(partA && ra == 31);
    const bool emitB = vb && rb < 32;
    uint32_t oc = ac;
    if (partA) oc = bbf_addmod(F, ac, pBc);
    const bool liveA = emitA && oc != 0u;
    const bool liveB = emitB && !partB;
    uint32_t mine = (liveA ? (1u << ra) : 0u) | (liveB ? (1u << rb) : 0u);
    const uint32_t live = __reduce_or_sync(BB_FULL, mine);
    const int nlive = __popc(live);
    if (no + nlive > cap) return -1;
    if (liveA) { int pos = no + __popc(live & ((1u << ra) - 1u)); Ok[pos] = ak; Oc[pos] = oc; }
    if (liveB) { int pos = no + __popc(live & ((1u << rb) - 1u)); Ok[pos] = bk; Oc[pos] = bc; }
    no += nlive;
    const int da = __popc(__ballot_sync(BB_FULL, emitA)), db = __popc(__ballot_sync(BB_FULL, emitB));
    if (da + db == 0) return -3;  // only reachable with unsorted (overflowed) keys
    ia += da; ib += db;
  }
  __syncwarp();
  return __any_sync(BB_FULL, (guard & K::g_all) != 0ull) ? -3 : no;
}

// The dividend h.  Its first two terms are always warp-uniform registers.  `mem` says whether the full list also sits
// in the slot's ping-pong scratch at half `buf`, offset `pos` (always true when n > 2).
struct Dividend {
  uint64_t k0, k1;
  uint32_t c0, c1;
  int n;
  int sug;  // sugar of h: max over the additions that built it of deg(multiplier) + sugar(operand), polynomials.cpp:150,198
  int loc;  // -1: registers only (n <= 2); else index of the lead term in the scratch (half * max_poly_terms + pos)
};

// a + b for lists of at most one term each, entirely in (uniform) registers
__device__ __forceinline__ void tiny_merge(const BBField& F, bool hasA, uint64_t ka, uint32_t ca, bool hasB, uint64_t kb,
                                           uint32_t cb, Dividend& o) {
  o.loc = -1;
  if (hasA && hasB) {
    if (ka == kb) {
      const uint32_t c = bbf_addmod(F, ca, cb);
      o.n = c ? 1 : 0; o.k0 = ka; o.c0 = c;
    } else {
      const bool af = ka < kb;
      o.k0 = af ? ka : kb; o.c0 = af ? ca : cb;
      o.k1 = af ? kb : ka; o.c1 = af ? cb : ca;
      o.n = 2;
    }
  } else if (hasA) { o.k0 = ka; o.c0 = ca; o.n = 1; }
  else if (hasB) { o.k0 = kb; o.c0 = cb; o.n = 1; }
  else o.n = 0;
}

// The remainder of a reduction in the two-term instantiations (TWO): at most two terms, warp-uniform registers, ascending
// key order.  In a binomial ideal every polynomial has at most two terms (DESIGN.md §3): the lead terms of an S-polynomial
// and of every reduction step cancel, leaving the two tails, and once a term has moved to the remainder the dividend has at
// most one term left.
struct Rem2 {
  uint64_t k0, k1;
  uint32_t c0, c1;
};

// h <- the n-term list a general merge left at the start of scratch half `buf`
__device__ __forceinline__ void dividend_from_scratch(const BBParams& P, const Env& e, Dividend& h, int n, int buf) {
  const uint64_t* hk = ENV_PTR(uint64_t, e, P, o_hkey) + (size_t)buf * P.max_poly_terms;
  const uint32_t* hc = ENV_PTR(uint32_t, e, P, o_hcoef) + (size_t)buf * P.max_poly_terms;
  h.n = n; h.loc = buf * P.max_poly_terms;
  if (n > 0) { h.k0 = hk[0]; h.c0 = hc[0]; }
  if (n > 1) { h.k1 = hk[1]; h.c1 = hc[1]; }
}

// ---------------------------------------------------------------------------------------------------- reduce
// Division algorithm of buchberger.cpp:24-49 on the dividend h.  Reducers are scanned IN ORDER (rlm[0..nR)), the
// first whose lead monomial divides LM(h) is used (h <- h - (LT h / LT f) f, steps++); otherwise LT(h) moves to the
// remainder, which is written to (rk, rc) [cap rcap].  Returns its length or -1 (scratch overflow) / -2 (remainder
// overflow) / -3 (exponent overflow detected).
// `sorted`: the reducer list is ascending in lead monomial, so the scan may stop at the first reducer whose lead
// monomial exceeds LM(h) (it and everything after it cannot divide); the count of examined lead monomials that
// feeds the traffic model stays the reference's (found + 1, or all of them).
// TWO: h and every reducer have at most two terms.  Only the register merge runs, and the remainder goes to *rem instead of
// (rk, rc), which stay untouched (the caller's update() writes it to the term arena); rcap still bounds its length.
template <int NV, bool TWO = false>
__device__ __forceinline__ int warp_reduce(const BBParams& P, Env& e, Dividend& h, const uint64_t* __restrict__ rlm,
                                           const uint32_t* __restrict__ ridx, int nR, bool sorted,
                                           uint64_t* __restrict__ rk, uint32_t* __restrict__ rc, int rcap, int& steps,
                                           Ctr& ct, Rem2* rem = nullptr) {
  typedef KL<NV> K;
  const BBField F = P.F;
  const int lane = bb_lane();
  const GHeadMem* gh = ENV_PTR(GHeadMem, e, P, o_ghead);
  int rlen = 0;
  steps = 0;
  while (h.n > 0) {
    const uint64_t lead = h.k0;
    int found = -1;
    uint32_t fidx = 0u;   // basis index of the divisor: loaded next to its lead monomial, one dependent load less per addition
#pragma unroll 1
    for (int base = 0; base < nR; base += 32) {
      const int r = base + lane;
      const uint64_t rl = r < nR ? rlm[r] : ~0ull;
      const uint32_t ix = r < nR ? ridx[r] : 0u;
      const uint32_t b = __ballot_sync(BB_FULL, r < nR && K::divides(rl, lead));
      if (b) { const int src = __ffs(b) - 1; found = base + src; fidx = __shfl_sync(BB_FULL, ix, src); break; }
      if (sorted && base + 32 < nR && __any_sync(BB_FULL, rl < lead)) break;  // larger lead monomials from here on (the last chunk ends the scan anyway)
    }
    ct.lms += (found >= 0) ? (found + 1) : nR;
    if (found >= 0) {
      const GHead f = load_head(gh + fidx);
      const uint32_t c = bbf_mulmod(F, h.c0, f.invlc);
      const uint32_t nc = F.p - c;              // c != 0
      const uint64_t adj = lead - f.lm;         // key(LM h / LM f) - bias
      {  // h.sug = max(h.sug, deg(LM h / LM f) + f.sug); term moves never raise it (sugar >= degree of every term)
        const int sf = (int)f.sug + (int)(uint32_t)(f.lm >> K::dshift) - (int)(uint32_t)(lead >> K::dshift);
        h.sug = sf > h.sug ? sf : h.sug;
      }
      ct.tread += (unsigned)h.n + f.len;
      if (TWO || (h.n <= 2 && f.len <= 2)) {
        const uint64_t kb = f.k1 + adj;
        const bool hasB = f.len == 2;
        if (hasB) e.guard |= kb;
        tiny_merge(F, h.n == 2, h.k1, h.c1, hasB, kb, bbf_mulmod(F, f.c1, nc), h);
        if (e.guard & K::g_all) return -3;  // garbage keys could otherwise keep the loop alive
      } else if constexpr (!TWO) {
        uint64_t* hk = ENV_PTR(uint64_t, e, P, o_hkey);
        uint32_t* hc = ENV_PTR(uint32_t, e, P, o_hcoef);
        if (h.loc < 0) {  // the register-resident dividend (n <= 2) goes to scratch half 0; only its tail is read
          h.loc = 0;
          if (lane == 0 && h.n == 2) { hk[1] = h.k1; hc[1] = h.c1; }
          __syncwarp();
        }
        const int ob = h.loc >= P.max_poly_terms ? 0 : 1;
        const size_t ho = (size_t)h.loc, oo = (size_t)ob * P.max_poly_terms;
        const uint64_t* tk = ENV_PTR(uint64_t, e, P, o_tkey);
        const uint32_t* tc = ENV_PTR(uint32_t, e, P, o_tcoef);
        const int n2 = warp_merge<NV>(F, hk + ho + 1, hc + ho + 1, h.n - 1, 1u, 0ull, tk + f.off + 1, tc + f.off + 1,
                                      (int)f.len - 1, nc, adj, hk + oo, hc + oo, P.max_poly_terms);
        if (n2 < 0) return n2;
        dividend_from_scratch(P, e, h, n2, ob);
      }
      ct.twrite += (unsigned)h.n;
      steps++;
    } else {
      if (rlen >= rcap) return -2;
      if constexpr (TWO) {
        if (rlen == 0) { rem->k0 = lead; rem->c0 = h.c0; }
        else { rem->k1 = lead; rem->c1 = h.c0; }
      } else {
        if (lane == 0) { rk[rlen] = lead; rc[rlen] = h.c0; }
      }
      rlen++;
      ct.moves++;
      h.n--; h.k0 = h.k1; h.c0 = h.c1;  // drop the lead term
      if constexpr (!TWO) {
        if (h.loc >= 0) {
          h.loc++;
          if (h.n > 1) {
            h.k1 = ENV_PTR(uint64_t, e, P, o_hkey)[h.loc + 1]; h.c1 = ENV_PTR(uint32_t, e, P, o_hcoef)[h.loc + 1];
          }
        }
      }
    }
  }
  if constexpr (!TWO) __syncwarp();
  return rlen;
}

// ---------------------------------------------------------------------------------------------------- update
// The fields of BBParams that update() reads.  warp_add_basis is one out-of-line copy, so `P` reaches it as a generic
// pointer into the kernel's parameter bank and every P.field would be a generic load (15 of them per call,
// profiles/README.md r2); every kernel that can reach it copies them to this block-shared record first (hot_init) and the
// function reads them with LDS at constant addresses.  -DBB_HOT_SHARED=0 reads P instead (A/B).
struct BBHot {
  int max_basis, max_pairs, elimination, sort_reducers;
  unsigned o_tkey, o_tcoef, o_lm, o_lscr, o_plcm, o_pairs, o_rlm, o_ridx, o_ghead, pad;
  const uint16_t* invtab;
};
#ifndef BB_HOT_SHARED
#define BB_HOT_SHARED 1
#endif
#if BB_HOT_SHARED
static __shared__ BBHot g_hot;
#define BB_HOT(P) g_hot
// every thread of the CTA, before anything else (contains a block barrier)
__device__ __forceinline__ void hot_init(const BBParams& P) {
  if (threadIdx.x == 0) {
    g_hot.max_basis = P.max_basis; g_hot.max_pairs = P.max_pairs; g_hot.elimination = P.elimination;
    g_hot.sort_reducers = P.sort_reducers; g_hot.o_tkey = P.o_tkey; g_hot.o_tcoef = P.o_tcoef; g_hot.o_lm = P.o_lm;
    g_hot.o_lscr = P.o_lscr; g_hot.o_plcm = P.o_plcm; g_hot.o_pairs = P.o_pairs; g_hot.o_rlm = P.o_rlm;
    g_hot.o_ridx = P.o_ridx; g_hot.o_ghead = P.o_ghead; g_hot.pad = 0u; g_hot.invtab = P.invtab;
  }
  __syncthreads();
}
#else
#define BB_HOT(P) (P)
__device__ __forceinline__ void hot_init(const BBParams&) {}
#endif

// Registers the polynomial stored at arena[off, off+len) (first two terms given in registers) as basis element
// m and runs update(G, P, f, elimination), buchberger.cpp:52-99, then the reducer-list insertion
// (upper_bound by lead monomial when sort_reducers: after every element whose lead monomial is <= the new one,
// buchberger.cpp:308-311 / 323-326).
// GebauerMoeller: (1) old (i,j) dropped iff LM f | lcm_ij and lcm_ij != lcm_if and lcm_ij != lcm_jf  (:63-70);
// (2-4) with L_i = lcm(LM_i, LM f):  (i,m) is emitted iff no L_j strictly divides L_i, no j < i has L_j == L_i,
// and no j with L_j == L_i is coprime to f.  This is exactly what the reference's ascending std::map sweep with
// the "not divisible by a previously kept lcm" filter, v[0] representative and none_of(coprime) test produces
// (:72-85): a kept lcm is a divisibility-minimal distinct lcm, and divisors always precede in grevlex order.
// (5) new pairs in ascending i (:86), appended after the survivors (:91-92).
// Every pair carries the key of its lcm (plcm), so step (1) and the selection strategies read one array.
// One out-of-line copy shared by step and reset.  Returns (emitted << 32) | new |P|, or -1 on pair-list overflow /
// -2 when the basis is full / -3 when an lcm's degree does not fit the packed layout; the caller bumps nG and nT.
// TWO: the polynomial (len <= 2 terms: lead key fk, coefficient c0, second term (k1, c1)) comes in registers and is written
// to arena[off, off+len) here, so update() starts without a dependent load.
template <int NV, bool TWO>
__device__ __forceinline__ long long add_basis_body(const BBParams& P, unsigned char* base, int m, int nP, int off, int len,
                                                    int sug, uint64_t fk, uint64_t k1, uint32_t c0, uint32_t c1) {
  typedef KL<NV> K;
  const auto& H = BB_HOT(P);
  const int lane = bb_lane();
  const uint32_t ltm = bb_lt_mask();
  if (m >= H.max_basis) return -2;
  base = bb_global(base);
  uint64_t* tk = reinterpret_cast<uint64_t*>(base + H.o_tkey) + off;
  uint32_t* tc = reinterpret_cast<uint32_t*>(base + H.o_tcoef) + off;
  if constexpr (!TWO) fk = tk[0];
  uint64_t* lm = reinterpret_cast<uint64_t*>(base + H.o_lm);
  uint64_t* lscr = reinterpret_cast<uint64_t*>(base + H.o_lscr);
  uint64_t* plcm = reinterpret_cast<uint64_t*>(base + H.o_plcm);
  uint32_t* pairs = reinterpret_cast<uint32_t*>(base + H.o_pairs);
  int emitted = 0;
  if (H.elimination == BB_ELIM_GEBAUERMOELLER && m <= 64) {
    // The common case (profiles/r01_v6: the sweep loop below was the largest single consumer of issue slots): with at
    // most 64 basis elements every lane keeps L_lane and L_{lane+32} in registers, so the peeling needs no memory at
    // all -- one candidate reduction and one two-register sweep per kept lcm.  Same algorithm as the general path.
    const int i0 = lane, i1 = lane + 32;
    const bool two = m > 32;   // warp-uniform: the second register of every lane is in use (1 call in 5 on the binomial workloads)
    const bool in0 = i0 < m, in1 = i1 < m;
    uint64_t v0 = 0ull, v1 = 0ull;
    bool cp0 = false, cp1 = false, ovf = false;
    if (in0) {
      const uint64_t l = lm[i0], le = K::lcm_exps(l, fk);
      const uint32_t dg = K::sum_fields(le);
      ovf |= dg > K::dmax;
      v0 = le | ((uint64_t)(K::dmax - dg) << K::dshift);
      cp0 = K::coprime(l, fk);
      lscr[i0] = v0;
    }
    if (in1) {
      const uint64_t l = lm[i1], le = K::lcm_exps(l, fk);
      const uint32_t dg = K::sum_fields(le);
      ovf |= dg > K::dmax;
      v1 = le | ((uint64_t)(K::dmax - dg) << K::dshift);
      cp1 = K::coprime(l, fk);
      lscr[i1] = v1;
    }
    if (__any_sync(BB_FULL, ovf)) return -3;
    __syncwarp();
    const uint64_t fe = fk & K::ex_mask;
    int w = 0;
#pragma unroll 1
    for (int b0 = 0; b0 < nP; b0 += 32) {   // step (1): old pairs, as in the general path
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
      if (keep) {
        const int pos = w + __popc(km & ltm);
        pairs[pos] = pr; plcm[pos] = pl;
      }
      w += __popc(km);
      __syncwarp();
    }
    nP = w;
    const uint64_t e0 = v0 & K::ex_mask, e1 = v1 & K::ex_mask;
    bool u0 = in0, u1 = in1, k0 = false, k1 = false;   // undecided / chosen for emission
    if (!two) {   // one lcm per lane: the same sweep without the second register (no code is shared on purpose: both loops are short)
      for (;;) {
        if (!__any_sync(BB_FULL, u0)) break;
        const uint32_t hi = __reduce_max_sync(BB_FULL, u0 ? (uint32_t)(v0 >> 32) : 0u);
        const bool c1 = u0 && (uint32_t)(v0 >> 32) == hi;
        const uint32_t lo = __reduce_max_sync(BB_FULL, c1 ? (uint32_t)v0 : 0u);
        const bool c2 = c1 && (uint32_t)v0 == lo;
        const int kidx = (int)__reduce_min_sync(BB_FULL, c2 ? (uint32_t)i0 : 0x7fffffffu);
        const uint64_t kk = (((uint64_t)hi << 32) | lo) & K::ex_mask;
        const bool d0 = u0 && ((((e0 | K::ge_mask) - kk) & K::ge_mask) == K::ge_mask);
        const bool grp_cop = __any_sync(BB_FULL, d0 && e0 == kk && cp0);
        u0 = u0 && !d0;
        if (!grp_cop) k0 = k0 || kidx == i0;
      }
    } else {
      for (;;) {
        const bool p1 = u1 && (!u0 || v1 > v0);          // this lane's larger undecided key; the lower index on a tie
        const uint64_t bk = p1 ? v1 : (u0 ? v0 : 0ull);
        if (!__any_sync(BB_FULL, u0 || u1)) break;
        const uint32_t hi = __reduce_max_sync(BB_FULL, (uint32_t)(bk >> 32));
        const bool c1 = (u0 || u1) && (uint32_t)(bk >> 32) == hi;
        const uint32_t lo = __reduce_max_sync(BB_FULL, c1 ? (uint32_t)bk : 0u);
        const bool c2 = c1 && (uint32_t)bk == lo;
        const int kidx = (int)__reduce_min_sync(BB_FULL, c2 ? (uint32_t)(p1 ? i1 : i0) : 0x7fffffffu);
        const uint64_t kk = (((uint64_t)hi << 32) | lo) & K::ex_mask;
        const bool d0 = u0 && ((((e0 | K::ge_mask) - kk) & K::ge_mask) == K::ge_mask);   // multiples of the killer, itself included
        const bool d1 = u1 && ((((e1 | K::ge_mask) - kk) & K::ge_mask) == K::ge_mask);
        const bool grp_cop = __any_sync(BB_FULL, (d0 && e0 == kk && cp0) || (d1 && e1 == kk && cp1));
        u0 = u0 && !d0; u1 = u1 && !d1;
        if (!grp_cop) { k0 = k0 || kidx == i0; k1 = k1 || kidx == i1; }
      }
    }
    const uint32_t km0 = __ballot_sync(BB_FULL, k0), km1 = two ? __ballot_sync(BB_FULL, k1) : 0u;
    const int cnt0 = __popc(km0), cnt1 = __popc(km1);
    if (nP + cnt0 + cnt1 > H.max_pairs) return -1;
    if (k0) { const int pos = nP + __popc(km0 & ltm); pairs[pos] = ((uint32_t)m << 16) | (uint32_t)i0; plcm[pos] = v0; }
    if (two && k1) { const int pos = nP + cnt0 + __popc(km1 & ltm); pairs[pos] = ((uint32_t)m << 16) | (uint32_t)i1; plcm[pos] = v1; }
    nP += cnt0 + cnt1; emitted = cnt0 + cnt1;
  } else if (H.elimination == BB_ELIM_GEBAUERMOELLER) {
    // lscr[i] = key of L_i = lcm(LM_i, LM f), for every basis element (the old-pair filter gathers from it)
    bool ovf = false;  // deg(L_i) must fit the degree field: bit 63 is a tag below, never a silently wrapped degree
#pragma unroll 1
    for (int i = lane; i < m; i += 32) {
      const uint64_t le = K::lcm_exps(lm[i], fk);
      const uint32_t dg = K::sum_fields(le);
      ovf |= dg > K::dmax;
      lscr[i] = le | ((uint64_t)(K::dmax - dg) << K::dshift);
    }
    if (__any_sync(BB_FULL, ovf)) return -3;
    __syncwarp();
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
    nP = w;
    // Steps (2)-(4) by peeling: the smallest remaining L (largest key; lowest index among equals = the group's
    // v[0]) cannot be strictly divided by anything still alive, so it is one of the reference's min_lcms.  It
    // kills every multiple (strict or equal), and its pair is emitted unless a member of its group is coprime to f.
    // One sweep over lscr per kept lcm instead of m sweeps: lscr[i] = key while undecided, 0 once dead,
    // key | 1<<63 once chosen for emission.
    uint64_t kk = 0ull, kkey = 0ull;   // exponents / key of the current killer
    int kidx = -1;
    for (;;) {
      uint64_t bk = 0ull; int bi = 0x7fffffff;
      uint32_t grp_cop = 0u;
#pragma unroll 1
      for (int b0 = 0; b0 < m; b0 += 32) {
        const int i = b0 + lane;
        uint64_t v = i < m ? lscr[i] : 0ull;
        bool und = v != 0ull && (long long)v > 0;  // undecided
        if (kidx >= 0) {
          const uint64_t ei = v & K::ex_mask;
          const bool eq = v != 0ull && ei == kk;    // the killer itself included
          if (und && ((((ei | K::ge_mask) - kk) & K::ge_mask) == K::ge_mask)) { lscr[i] = 0ull; und = false; }
          bool cop = false;
          if (eq) cop = K::coprime(lm[i], fk);
          grp_cop |= __ballot_sync(BB_FULL, cop);
        }
        if (und && v > bk) { bk = v; bi = i; }  // ascending i per lane: first occurrence kept on ties
      }
      if (kidx >= 0 && lane == 0) lscr[kidx] = grp_cop ? 0ull : (kkey | (1ull << 63));
      if (!__any_sync(BB_FULL, bk != 0ull)) break;  // nothing undecided
      // next killer: largest key, lowest index among equals
      const uint32_t hi = __reduce_max_sync(BB_FULL, (uint32_t)(bk >> 32));
      const bool c1 = (uint32_t)(bk >> 32) == hi;
      const uint32_t lo = __reduce_max_sync(BB_FULL, c1 ? (uint32_t)bk : 0u);
      const bool c2 = c1 && (uint32_t)bk == lo;
      kidx = (int)__reduce_min_sync(BB_FULL, c2 ? (uint32_t)bi : 0x7fffffffu);
      kkey = ((uint64_t)hi << 32) | lo;
      kk = kkey & K::ex_mask;
      if (lane == 0) lscr[kidx] |= (1ull << 63);  // decided: out of the undecided set while it sweeps
      __syncwarp();
    }
    __syncwarp();
#pragma unroll 1
    for (int b0 = 0; b0 < m; b0 += 32) {
      const int i = b0 + lane;
      const uint64_t v = i < m ? lscr[i] : 0ull;
      const bool keep = (long long)v < 0;
      const uint32_t km = __ballot_sync(BB_FULL, keep);
      const int cnt = __popc(km);
      if (nP + cnt > H.max_pairs) return -1;
      if (keep) {
        const int pos = nP + __popc(km & ltm);
        pairs[pos] = ((uint32_t)m << 16) | (uint32_t)i;
        plcm[pos] = v & ~(1ull << 63);
      }
      nP += cnt; emitted += cnt;
    }
  } else {
#pragma unroll 1
    for (int b0 = 0; b0 < m; b0 += 32) {
      const int i = b0 + lane;
      bool keep = i < m;
      const uint64_t li = keep ? lm[i] : 0ull;
      if (keep && H.elimination == BB_ELIM_LCM) keep = !K::coprime(li, fk);  // :58-62
      const uint32_t km = __ballot_sync(BB_FULL, keep);
      const int cnt = __popc(km);
      if (nP + cnt > H.max_pairs) return -1;
      if (keep) {
        const int pos = nP + __popc(km & ltm);
        pairs[pos] = ((uint32_t)m << 16) | (uint32_t)i;
        plcm[pos] = K::key_from_exps(K::lcm_exps(li, fk));
      }
      nP += cnt; emitted += cnt;
    }
  }
  // reducer list
  uint64_t* rlm = reinterpret_cast<uint64_t*>(base + H.o_rlm);
  uint32_t* ridx = reinterpret_cast<uint32_t*>(base + H.o_ridx);
  int pos = m;
  if (H.sort_reducers && m <= 64) {   // both halves of the list in registers: count, then shift by one, no read-after-write hazard
    const int i0 = lane, i1 = lane + 32;
    uint64_t r0 = 0ull, r1 = 0ull; uint32_t x0 = 0u, x1 = 0u;
    const bool two = m > 32;
    if (i0 < m) { r0 = rlm[i0]; x0 = ridx[i0]; }
    if (two && i1 < m) { r1 = rlm[i1]; x1 = ridx[i1]; }
    // reducers with LM <= new LM  <=>  key >= new key; the list is sorted, so they are a prefix
    pos = __popc(__ballot_sync(BB_FULL, i0 < m && r0 >= fk));
    if (two) pos += __popc(__ballot_sync(BB_FULL, i1 < m && r1 >= fk));
    __syncwarp();
    if (i0 < m && i0 >= pos) { rlm[i0 + 1] = r0; ridx[i0 + 1] = x0; }
    if (two && i1 < m && i1 >= pos) { rlm[i1 + 1] = r1; ridx[i1 + 1] = x1; }
    __syncwarp();
  } else if (H.sort_reducers) {
    int cnt = 0;  // reducers with LM <= new LM  <=>  key >= new key
#pragma unroll 1
    for (int b0 = 0; b0 < m; b0 += 32) {
      const int r = b0 + lane;
      cnt += __popc(__ballot_sync(BB_FULL, r < m && rlm[r] >= fk));
    }
    pos = cnt;
#pragma unroll 1
    for (int hi = m; hi > pos; hi -= 32) {
      const int lo = hi - 32 > pos ? hi - 32 : pos;
      const int idx = lo + lane;
      const bool v = idx < hi;
      uint64_t k = 0; uint32_t ix = 0;
      if (v) { k = rlm[idx]; ix = ridx[idx]; }
      __syncwarp();
      if (v) { rlm[idx + 1] = k; ridx[idx + 1] = ix; }
      __syncwarp();
    }
  }
  if (lane == 0) {
    rlm[pos] = fk; ridx[pos] = (uint32_t)m;
    lm[m] = fk;
    GHeadMem* g = reinterpret_cast<GHeadMem*>(base + H.o_ghead) + m;
    if constexpr (TWO) {
      tk[0] = fk; tc[0] = c0;
      if (len > 1) { tk[1] = k1; tc[1] = c1; }
      else { k1 = 0ull; c1 = 0u; }
    }
    const uint32_t inv = bb_global(H.invtab)[TWO ? c0 : tc[0]];  // 1/LC: one table load instead of a 15-step power ladder
    if constexpr (!TWO) {
      k1 = len > 1 ? tk[1] : 0ull;
      c1 = len > 1 ? tc[1] : 0u;
    }
    reinterpret_cast<uint4*>(g)[0] = make_uint4((uint32_t)fk, (uint32_t)(fk >> 32), (uint32_t)k1, (uint32_t)(k1 >> 32));
    reinterpret_cast<uint4*>(g)[1] = make_uint4(inv | (c1 << 16), (uint32_t)sug, (uint32_t)off, (uint32_t)len);
  }
  __syncwarp();
  return ((long long)emitted << 32) | (long long)nP;
}
// the polynomial already sits at arena[off, off+len)
template <int NV>
__device__ BB_ADD_BASIS_INLINE long long warp_add_basis(const BBParams& P, unsigned char* base, int m, int nP, int off, int len,
                                                        int sug) {
  return add_basis_body<NV, false>(P, base, m, nP, off, len, sug, 0ull, 0ull, 0u, 0u);
}
// two-term instantiation: the polynomial in registers, see add_basis_body.  Inlined: its one call site is the two-term
// k_run's warp_step, and without the call's register save / restore that kernel spills 248 instead of 380 bytes at its
// 64-register cap (profiles/README.md, "Two-term runner at 32 warps per SM")
template <int NV>
__device__ __forceinline__ long long warp_add_basis(const BBParams& P, unsigned char* base, int m, int nP, int off, int len,
                                                        int sug, uint64_t fk, uint64_t k1, uint32_t c0, uint32_t c1) {
  return add_basis_body<NV, true>(P, base, m, nP, off, len, sug, fk, k1, c0, c1);
}

// ---------------------------------------------------------------------------------------------------- step
// Removes row `row` from the pair list keeping order (buchberger.cpp:319) and returns the pair ((j << 16) | i) and the
// cached key of its lcm.  Caller guarantees 0 <= row < |P|.
__device__ __forceinline__ void warp_take_pair(const BBParams& P, Env& e, int row, uint32_t& pr, uint64_t& gam) {
  const int lane = bb_lane();
  uint32_t* pairs = ENV_PTR(uint32_t, e, P, o_pairs);
  uint64_t* plcm = ENV_PTR(uint64_t, e, P, o_plcm);
  pr = pairs[row];
  gam = plcm[row];  // key of lcm(LM f, LM g), computed when the pair was created
  __syncwarp();
#pragma unroll 1
  for (int b0 = row; b0 < e.nP - 1; b0 += 32) {
    const int idx = b0 + lane;
    const bool v = idx < e.nP - 1;
    uint32_t x = 0u; uint64_t y = 0ull;
    if (v) { x = pairs[idx + 1]; y = plcm[idx + 1]; }
    __syncwarp();
    if (v) { pairs[idx] = x; plcm[idx] = y; }
  }
  e.nP--;
}

// BuchbergerEnv::step for the pair in row `row` of P (LeadMonomialsEnv::step(int), buchberger.cpp:398-408 ->
// :318-329): erase the pair, s = spoly(G[i], G[j]) (:18-21), (r, steps) = reduce(s, G_), if r != 0 update + sorted
// insert.  Returns the number of polynomial additions 1 + steps (reward = -(1+steps) under Additions, -1 under
// Reductions).  `pair` receives (j << 16) | i, or 0xffffffff for a bad action.
// TWO: every polynomial of the environment has at most two terms (binomial ideals): no general merge, no scratch, and the
// remainder reaches update() in registers.  Same results and counters as the general instantiation.
template <int NV, bool TWO = false>
__device__ __forceinline__ int warp_step(const BBParams& P, Env& e, int row, uint32_t& pair, Ctr& ct) {
  typedef KL<NV> K;
  const BBField F = P.F;
  if ((unsigned)row >= (unsigned)e.nP) { e.status = BB_STATUS_BAD_ACTION; pair = 0xffffffffu; return 0; }
  uint32_t pr; uint64_t gam;
  warp_take_pair(P, e, row, pr, gam);
  const int i = pr & 0xffffu, j = pr >> 16;
  pair = pr;  // (j << 16) | i; never 0xffffffff because i < j
  // S-polynomial: lead terms cancel exactly, so s = (gamma/LT f) tail(f) - (gamma/LT g) tail(g)
  const GHeadMem* gh = ENV_PTR(GHeadMem, e, P, o_ghead);
  const GHead hf = load_head(gh + i), hg = load_head(gh + j);
  e.guard |= gam;
  ct.tread += hf.len + hg.len;
  Dividend h;
  h.k0 = h.k1 = 0; h.c0 = h.c1 = 0; h.n = 0; h.loc = -1;
  {  // sugar of the S-polynomial: max(deg(gamma / LM f) + sug f, deg(gamma / LM g) + sug g)
    const int cg0 = (int)(uint32_t)(gam >> K::dshift);
    const int sf = (int)hf.sug + (int)(uint32_t)(hf.lm >> K::dshift) - cg0, sg = (int)hg.sug + (int)(uint32_t)(hg.lm >> K::dshift) - cg0;
    h.sug = sf > sg ? sf : sg;
  }
  const uint64_t adjf = gam - hf.lm, adjg = gam - hg.lm;
  const uint32_t cg = F.p - hg.invlc;  // -(1/LC g), invlc != 0
  if (TWO || (hf.len <= 2 && hg.len <= 2)) {
    const uint64_t ka = hf.k1 + adjf, kb = hg.k1 + adjg;
    const bool hasA = hf.len == 2, hasB = hg.len == 2;
    if (hasA) e.guard |= ka;
    if (hasB) e.guard |= kb;
    tiny_merge(F, hasA, ka, bbf_mulmod(F, hf.c1, hf.invlc), hasB, kb, bbf_mulmod(F, hg.c1, cg), h);
  } else if constexpr (!TWO) {
    const uint64_t* tk = ENV_PTR(uint64_t, e, P, o_tkey);
    const uint32_t* tc = ENV_PTR(uint32_t, e, P, o_tcoef);
    const int n = warp_merge<NV>(F, tk + hf.off + 1, tc + hf.off + 1, (int)hf.len - 1, hf.invlc, adjf, tk + hg.off + 1,
                                 tc + hg.off + 1, (int)hg.len - 1, cg, adjg, ENV_PTR(uint64_t, e, P, o_hkey),
                                 ENV_PTR(uint32_t, e, P, o_hcoef), P.max_poly_terms);
    if (n == -1) { e.status = BB_STATUS_OVERFLOW_SCRATCH; return 1; }
    if (n < 0) { e.status = BB_STATUS_OVERFLOW_EXPONENT; return 1; }
    dividend_from_scratch(P, e, h, n, 0);
  }
  if (e.guard & K::g_all) { e.status = BB_STATUS_OVERFLOW_EXPONENT; return 1; }
  ct.twrite += (unsigned)h.n;
  int steps = 0;
  Rem2 rem;
  const int rlen = warp_reduce<NV, TWO>(P, e, h, ENV_PTR(uint64_t, e, P, o_rlm), ENV_PTR(uint32_t, e, P, o_ridx), e.nG,
                                        P.sort_reducers != 0, ENV_PTR(uint64_t, e, P, o_tkey) + e.nT,
                                        ENV_PTR(uint32_t, e, P, o_tcoef) + e.nT, P.max_terms - e.nT, steps, ct, &rem);
  if (rlen < 0 || (e.guard & K::g_all)) {   // one test on the hot path; which fault it was is sorted out here
    e.status = rlen == -1 ? BB_STATUS_OVERFLOW_SCRATCH : (rlen == -2 ? BB_STATUS_OVERFLOW_TERMS : BB_STATUS_OVERFLOW_EXPONENT);
    return 1 + steps;
  }
  if (rlen > 0) {
    ct.upb += (unsigned)e.nG; ct.upp += (unsigned)e.nP;
    long long r;
    if constexpr (TWO) r = warp_add_basis<NV>(P, e.base, e.nG, e.nP, e.nT, rlen, h.sug, rem.k0, rem.k1, rem.c0, rem.c1);
    else r = warp_add_basis<NV>(P, e.base, e.nG, e.nP, e.nT, rlen, h.sug);
    if (r < 0) {
      e.status = (r == -1) ? BB_STATUS_OVERFLOW_PAIRS : (r == -2 ? BB_STATUS_OVERFLOW_BASIS : BB_STATUS_OVERFLOW_EXPONENT);
      return 1 + steps;
    }
    e.nP = (int)(r & 0xffffffffll);
    ct.upp += (unsigned)(r >> 32);
    e.nG++; e.nT += rlen;
  }
  if (e.nP == 0) e.status = BB_STATUS_DONE;
  return 1 + steps;
}

// ---------------------------------------------------------------------------------------------------- select
// Pair selection, buchberger.cpp:160-241.  Every comparator ends in (j, i), and P is always sorted by (j, i), so
// "first minimal element" is the lowest row among ties for the ascending strategies (First, Degree, Normal, Sugar)
// and the HIGHEST row among ties for the reversed ones (Last, Codegree, Strange, Spice: min_element under '>').
// Reads only the cached lcm keys, except Sugar / Spice which gather the two head records of each pair.

// argmax of a 64-bit value with an index tie-break (low: lowest index wins, else highest); lanes without a
// candidate pass idx = 0xffffffff
__device__ __forceinline__ int warp_argmax64(uint64_t v, uint32_t idx, bool low) {
  const bool has = idx != 0xffffffffu;
  const uint32_t hi = __reduce_max_sync(BB_FULL, has ? (uint32_t)(v >> 32) : 0u);
  const bool c1 = has && (uint32_t)(v >> 32) == hi;
  const uint32_t lo = __reduce_max_sync(BB_FULL, c1 ? (uint32_t)v : 0u);
  const bool c2 = c1 && (uint32_t)v == lo;
  return low ? (int)__reduce_min_sync(BB_FULL, c2 ? idx : 0xffffffffu) : (int)__reduce_max_sync(BB_FULL, c2 ? idx : 0u);
}

// sugar of pair (i, j) with lcm key l: max(sug_i + deg(l / LM_i), sug_j + deg(l / LM_j))   (buchberger.cpp:189-192)
template <int NV>
__device__ __forceinline__ int pair_sugar(const GHeadMem* gh, uint32_t pr, uint64_t l) {
  typedef KL<NV> K;
  const GHeadMem* a = gh + (pr & 0xffffu); const GHeadMem* b = gh + (pr >> 16);
  const int cl = (int)(uint32_t)(l >> K::dshift);
  const int sa = (int)a->sug + (int)(uint32_t)(a->lm >> K::dshift) - cl, sb = (int)b->sug + (int)(uint32_t)(b->lm >> K::dshift) - cl;
  return sa > sb ? sa : sb;
}

// the strategies outside the benchmarked three: one out-of-line copy
template <int NV>
__device__ __noinline__ int warp_select_rare(const BBParams& P, unsigned char* base, int nP, int strategy, uint32_t* rng) {
  typedef KL<NV> K;
  const int lane = bb_lane();
  base = bb_global(base);
  const uint64_t* plcm = reinterpret_cast<const uint64_t*>(base + P.o_plcm);
  if (strategy == BB_SELECT_RANDOM) {  // choice(): uniform_int_distribution<>(0, |P|-1)(rng), ideals.h:68-73
    uint32_t x = *rng;                        // rng: shared or global memory, one word per environment
    const int r = rng_uniform(x, 0, nP - 1);  // every lane runs the same stream
    __syncwarp();
    if (lane == 0) *rng = x;
    __syncwarp();
    return r;
  }
  if (strategy == BB_SELECT_LAST) return nP - 1;
  if (strategy == BB_SELECT_CODEGREE) {  // largest degree == smallest complemented-degree field; highest row on ties
    uint32_t best = 0u;
#pragma unroll 1
    for (int idx = lane; idx < nP; idx += 32) {
      const uint32_t v = ((K::dmax - (uint32_t)(plcm[idx] >> K::dshift)) << 16) | (uint32_t)idx;
      best = v > best ? v : best;
    }
    return (int)(__reduce_max_sync(BB_FULL, best) & 0xffffu);
  }
  if (strategy == BB_SELECT_STRANGE) {  // largest lcm in grevlex == SMALLEST key; highest row on ties
    uint64_t bk = 0; uint32_t bi = 0xffffffffu;
#pragma unroll 1
    for (int idx = lane; idx < nP; idx += 32) {
      const uint64_t k = ~plcm[idx];
      if (k >= bk) { bk = k; bi = (uint32_t)idx; }  // ascending idx per lane: last occurrence kept on ties
    }
    return warp_argmax64(bk, bi, false);
  }
  // Sugar: min (sugar, lcm, j, i); Spice: max of the same tuple
  const bool spice = strategy == BB_SELECT_SPICE;
  const uint32_t* pairs = reinterpret_cast<const uint32_t*>(base + P.o_pairs);
  const GHeadMem* gh = reinterpret_cast<const GHeadMem*>(base + P.o_ghead);
  int bs = spice ? -1 : 0x7fffffff;
#pragma unroll 1
  for (int idx = lane; idx < nP; idx += 32) {
    const int sg = pair_sugar<NV>(gh, pairs[idx], plcm[idx]);
    bs = spice ? (sg > bs ? sg : bs) : (sg < bs ? sg : bs);
  }
  bs = spice ? (int)__reduce_max_sync(BB_FULL, (uint32_t)(bs + 1)) - 1 : (int)__reduce_min_sync(BB_FULL, (uint32_t)bs);
  uint64_t bk = 0; uint32_t bi = 0xffffffffu;
#pragma unroll 1
  for (int idx = lane; idx < nP; idx += 32) {
    const uint64_t l = plcm[idx];
    if (pair_sugar<NV>(gh, pairs[idx], l) != bs) continue;
    const uint64_t k = spice ? ~l : l;  // Sugar: smallest lcm == largest key; Spice: largest lcm == smallest key
    if (bi == 0xffffffffu || (spice ? k >= bk : k > bk)) { bk = k; bi = (uint32_t)idx; }
  }
  return warp_argmax64(bk, bi, !spice);
}

template <int NV>
__device__ __forceinline__ int warp_select(const BBParams& P, const Env& e, int strategy, uint32_t* rng) {
  typedef KL<NV> K;
  const int lane = bb_lane();
  if (strategy == BB_SELECT_FIRST) return 0;
  if (strategy > BB_SELECT_NORMAL) return warp_select_rare<NV>(P, e.base, e.nP, strategy, rng);
  if (e.nP <= 1) return 0;
  const uint64_t* plcm = ENV_PTR(uint64_t, e, P, o_plcm);
  if (strategy == BB_SELECT_DEGREE) {
    // smallest degree == largest complemented-degree field; lowest row on ties
    uint32_t best = 0u;
#pragma unroll 1
    for (int idx = lane; idx < e.nP; idx += 32) {
      const uint32_t v = ((uint32_t)(plcm[idx] >> K::dshift) << 16) | (0xffffu - (uint32_t)idx);
      best = v > best ? v : best;
    }
    best = __reduce_max_sync(BB_FULL, best);
    return (int)(0xffffu - (best & 0xffffu));
  }
  // Normal: smallest lcm in grevlex == LARGEST key; lowest row on ties
  uint64_t bk = 0; uint32_t bi = 0xffffffffu;
#pragma unroll 1
  for (int idx = lane; idx < e.nP; idx += 32) {
    const uint64_t k = plcm[idx];
    if (k > bk) { bk = k; bi = (uint32_t)idx; }  // strided ascending idx: first occurrence kept on ties
  }
  return warp_argmax64(bk, bi, true);
}

// ---------------------------------------------------------------------------------------------------- observe
// Row r of the state matrix = first k exponent vectors of G[i] then of G[j], zero padded
// (lead_monomials_vector, buchberger.cpp:354-370; rows in P order, :402-406); rows [|P|, pmax) are -1.
template <int NV>
__device__ __forceinline__ void warp_observe(const BBParams& P, const Env& e, int32_t* obs, int pmax, Ctr& ct) {
  typedef KL<NV> K;
  const int lane = bb_lane();
  const int nv = P.obs_nv;   // == NV except under bb_set_obs_nvars (the C++ FixedIdealGenerator::nvars quirk, ideals.cpp:146-154)
  const int k = P.k, cols = P.cols, half = nv * k;
  const int rows = e.nP < pmax ? e.nP : pmax;
  const uint32_t* pairs = ENV_PTR(uint32_t, e, P, o_pairs);
  const GHeadMem* gh = ENV_PTR(GHeadMem, e, P, o_ghead);
  const uint64_t* tk = ENV_PTR(uint64_t, e, P, o_tkey);
  // one lane per (row, side): 16 rows per pass; the lane loads its polynomial's head record once and writes the k * nv
  // exponents of that half row, so consecutive lanes write consecutive half rows (no division per element, two
  // dependent loads per half row instead of three per element)
  const int side = lane & 1;
#pragma unroll 1
  for (int r0 = 0; r0 < rows; r0 += 16) {
    const int row = r0 + (lane >> 1);
    if (row < rows) {
      const uint32_t pr = pairs[row];
      const GHead g = load_head(gh + (side ? (pr >> 16) : (pr & 0xffffu)));
      int32_t* o = obs + (size_t)row * cols + side * half;
#pragma unroll 1
      for (int t = 0; t < k; t++) {
        const bool have = t < (int)g.len;
        const uint64_t key = t == 0 ? g.lm : (t == 1 ? g.k1 : (have ? tk[g.off + t] : 0ull));
        for (int v = 0; v < nv; v++) o[t * nv + v] = have ? (int32_t)K::exp(key, v) : 0;
      }
    }
  }
  // rows [|P|, pmax) are -1: 16-byte stores where the row pitch allows it
  const int live = rows * cols, total = pmax * cols;
  if (((cols & 3) == 0) && ((reinterpret_cast<uintptr_t>(obs) & 15) == 0)) {
    int4* o4 = reinterpret_cast<int4*>(obs + live);
    const int n4 = (total - live) >> 2;
    const int4 m1 = make_int4(-1, -1, -1, -1);
    for (int x = lane; x < n4; x += 32) o4[x] = m1;
  } else {
    for (int x = live + lane; x < total; x += 32) obs[x] = -1;
  }
  ct.obs += (unsigned)rows;
}

// ---------------------------------------------------------------------------------------------------- generator
// RandomBinomialIdealGenerator::next (ideals.cpp:168-201), executed by lane 0 into the slot's staging area.
// Returns false if 1000 trials fail (the reference throws).
__device__ __forceinline__ bool gen_binomial_ideal(const BBParams& P, int slot, uint32_t& x) {
  const BBDist& D = P.dist;
  uint64_t* ik = P.in_key + (size_t)slot * P.max_gen_terms;
  uint32_t* ic = P.in_coef + (size_t)slot * P.max_gen_terms;
  int* io = P.in_off + (size_t)slot * (P.max_gens + 1);
  io[0] = 0;
  for (int i = 0; i < D.s; i++) {
    const uint32_t c = D.pure ? (P.F.p - 1u) : (uint32_t)rng_uniform(x, 1, (int)P.F.p - 1);
    int d1, d2;
    if (D.homogeneous) d1 = d2 = rng_degree(D, x);
    else { d1 = rng_degree(D, x); d2 = rng_degree(D, x); }
    const int o1 = D.basis_off[d1], n1 = D.basis_off[d1 + 1] - o1, o2 = D.basis_off[d2], n2 = D.basis_off[d2 + 1] - o2;
    bool ok = false;
    for (int trials = 0; trials < 1000 && !ok; trials++) {
      const uint64_t m1 = D.basis[o1 + rng_uniform(x, 0, n1 - 1)];
      const uint64_t m2 = D.basis[o2 + rng_uniform(x, 0, n2 - 1)];
      if (m1 != m2) {  // larger monomial (smaller key) leads with coefficient 1
        const uint64_t hi = m1 < m2 ? m1 : m2, lo = m1 < m2 ? m2 : m1;
        ik[2 * i] = hi; ic[2 * i] = 1u; ik[2 * i + 1] = lo; ic[2 * i + 1] = c;
        ok = true;
      }
    }
    if (!ok) return false;
    io[i + 1] = 2 * (i + 1);
  }
  P.in_np[slot] = D.s;
  return true;
}

// RandomIdealGenerator::next (ideals.cpp:214-231), executed by lane 0 into the slot's staging area: per generator
// terms = 2 + Poisson(lam) draws of (coefficient, monomial of the current degree) summed into f (equal monomials add,
// a zero sum drops out: Polynomial operator+, polynomials.cpp:148-177), a fresh degree after every term unless homog,
// then f / LC(f).  libstdc++'s poisson_distribution for mean < 12 multiplies canonicals until the product falls to
// exp(-mean) (bits/random.tcc, the branch without _GLIBCXX_USE_C99_MATH_TR1's rejection method).
// Returns 1, 0 if a polynomial cancelled to zero (f.LC() of an empty polynomial is undefined behaviour in the
// reference), -1 if the ideal does not fit max_gen_terms.
__device__ __forceinline__ int gen_random_ideal(const BBParams& P, int slot, uint32_t& x) {
  const BBDist& D = P.dist;
  const BBField F = P.F;
  uint64_t* ik = P.in_key + (size_t)slot * P.max_gen_terms;
  uint32_t* ic = P.in_coef + (size_t)slot * P.max_gen_terms;
  int* io = P.in_off + (size_t)slot * (P.max_gens + 1);
  io[0] = 0;
  int nt = 0;
  for (int i = 0; i < D.s; i++) {
    int cnt = 0;
    double prod = 1.0;
    do { prod = __dmul_rn(prod, rng_canonical(x)); cnt++; } while (prod > D.lm_thr);
    const int terms = 2 + (cnt - 1);
    int d = rng_degree(D, x);
    uint64_t* fk = ik + nt; uint32_t* fc = ic + nt;
    int len = 0;
    for (int j = 0; j < terms; j++) {
      const uint32_t c = (uint32_t)rng_uniform(x, 1, (int)F.p - 1);
      const int o = D.basis_off[d], nb = D.basis_off[d + 1] - o;
      const uint64_t m = D.basis[o + rng_uniform(x, 0, nb - 1)];
      int pos = 0;
      while (pos < len && fk[pos] < m) pos++;
      if (pos < len && fk[pos] == m) {
        const uint32_t sum = bbf_addmod(F, fc[pos], c);
        if (sum) fc[pos] = sum;
        else { for (int t = pos; t + 1 < len; t++) { fk[t] = fk[t + 1]; fc[t] = fc[t + 1]; } len--; }
      } else {
        if (nt + len + 1 > P.max_gen_terms) return -1;
        for (int t = len; t > pos; t--) { fk[t] = fk[t - 1]; fc[t] = fc[t - 1]; }
        fk[pos] = m; fc[pos] = c; len++;
      }
      if (!D.homogeneous) d = rng_degree(D, x);
    }
    if (len == 0) return 0;
    const uint32_t inv = P.invtab[fc[0]];
    for (int t = 0; t < len; t++) fc[t] = bbf_mulmod(F, fc[t], inv);
    nt += len;
    io[i + 1] = nt;
  }
  P.in_np[slot] = D.s;
  return 1;
}

// The same generator with one lane per generator.  minstd_rand0 is a pure multiplicative congruence, so the state
// before generator g is a^(g * draws_per_generator) * x provided every earlier generator consumed the nominal number
// of draws (1 coefficient + 2 per degree + 1 per monomial pick).  It does unless a uniform_int draw was rejected
// (p < 1e-5) or the two monomials coincided (p ~ 0.2 %): every lane checks that its own state advanced by exactly the
// nominal power, and one deviation anywhere sends the whole ideal back to the serial restatement above.  x must be
// warp-uniform; returns false without touching it when the serial path has to run.
__device__ __forceinline__ uint32_t rng_mulmod(uint32_t a, uint32_t b) {
  const unsigned long long pr = (unsigned long long)a * b;              // < 2^62
  unsigned long long r = (pr & 0x7fffffffULL) + (pr >> 31);             // 2^31 == 1 (mod 2^31 - 1);  < 2^32
  uint32_t q = (uint32_t)(r & 0x7fffffffULL) + (uint32_t)(r >> 31);     // <= 2^31
  if (q >= 2147483647u) q -= 2147483647u;
  return q;
}
__device__ __forceinline__ bool gen_binomial_ideal_warp(const BBParams& P, int slot, uint32_t& x) {
  const BBDist& D = P.dist;
  if (D.s > 32) return false;
  const int lane = bb_lane();
  const int nominal = (D.pure ? 0 : 1) + (D.ncp < 2 ? 0 : (D.homogeneous ? 2 : 4)) + 2;
  uint32_t an = 1u;                                   // a^nominal
  for (int k = 0; k < nominal; k++) rng_next(an);
  uint32_t mult = 1u, sq = an;                        // a^(nominal * lane)
  for (int e = lane; e; e >>= 1) { if (e & 1) mult = rng_mulmod(mult, sq); sq = rng_mulmod(sq, sq); }
  uint32_t y = rng_mulmod(x, mult);
  bool fine = true;
  uint64_t hi = 0ull, lo = 0ull; uint32_t c = 0u;
  if (lane < D.s) {
    const uint32_t expect = rng_mulmod(y, an);
    c = D.pure ? (P.F.p - 1u) : (uint32_t)rng_uniform(y, 1, (int)P.F.p - 1);
    int d1, d2;
    if (D.homogeneous) d1 = d2 = rng_degree(D, y);
    else { d1 = rng_degree(D, y); d2 = rng_degree(D, y); }
    const int o1 = D.basis_off[d1], n1 = D.basis_off[d1 + 1] - o1, o2 = D.basis_off[d2], n2 = D.basis_off[d2 + 1] - o2;
    const uint64_t m1 = D.basis[o1 + rng_uniform(y, 0, n1 - 1)];
    const uint64_t m2 = D.basis[o2 + rng_uniform(y, 0, n2 - 1)];
    hi = m1 < m2 ? m1 : m2; lo = m1 < m2 ? m2 : m1;
    fine = m1 != m2 && y == expect;
  }
  if (!__all_sync(BB_FULL, fine)) return false;
  uint64_t* ik = P.in_key + (size_t)slot * P.max_gen_terms;
  uint32_t* ic = P.in_coef + (size_t)slot * P.max_gen_terms;
  int* io = P.in_off + (size_t)slot * (P.max_gens + 1);
  if (lane < D.s) {
    ik[2 * lane] = hi; ic[2 * lane] = 1u; ik[2 * lane + 1] = lo; ic[2 * lane + 1] = c;
    io[lane + 1] = 2 * (lane + 1);
  }
  if (lane == 0) { io[0] = 0; P.in_np[slot] = D.s; }
  x = __shfl_sync(BB_FULL, y, D.s - 1);
  return true;
}

// ---------------------------------------------------------------------------------------------------- reset
// BuchbergerEnv::reset (buchberger.cpp:299-315) from staged ideal `src_slot` into slot `slot`: generators are added
// one by one through update() and into the reducer list.  sort_input orders them by ascending lead monomial first
// (stable).  Leaves (nG, nP, nT, status) in e.
template <int NV>
__device__ __forceinline__ void warp_load_ideal(const BBParams& P, int src_slot, Env& e, Ctr& ct) {
  const int lane = bb_lane();
  const uint64_t* ik = P.in_key + (size_t)src_slot * P.max_gen_terms;
  const uint32_t* ic = P.in_coef + (size_t)src_slot * P.max_gen_terms;
  const int* io = P.in_off + (size_t)src_slot * (P.max_gens + 1);
  const int np = P.in_np[src_slot];
  uint64_t* tk = ENV_PTR(uint64_t, e, P, o_tkey);
  uint32_t* tc = ENV_PTR(uint32_t, e, P, o_tcoef);
  e.nG = 0; e.nP = 0; e.nT = 0; e.guard = 0;
  e.status = BB_STATUS_RUNNING;
  for (int q = 0; q < np; q++) {
    int src = q;
    if (P.sort_input) {  // the generator whose stable ascending-LM rank is q
      int mine = -1;
      for (int g = lane; g < np; g += 32) {
        const uint64_t kg = ik[io[g]];
        int rank = 0;
        for (int o = 0; o < np; o++) { const uint64_t ko = ik[io[o]]; rank += (ko > kg) || (ko == kg && o < g); }
        if (rank == q) mine = g;
      }
      const uint32_t b = __ballot_sync(BB_FULL, mine >= 0);
      src = __shfl_sync(BB_FULL, mine, __ffs(b) - 1);
    }
    const int off = io[src], len = io[src + 1] - off;
    if (e.nT + len > P.max_terms) { e.status = BB_STATUS_OVERFLOW_TERMS; return; }
#pragma unroll 1
    for (int t = lane; t < len; t += 32) { tk[e.nT + t] = ik[off + t]; tc[e.nT + t] = ic[off + t]; }
    __syncwarp();
    ct.upb += (unsigned)e.nG; ct.upp += (unsigned)e.nP;
    const long long r = warp_add_basis<NV>(P, e.base, e.nG, e.nP, e.nT, len,
                                               (int)KL<NV>::deg(ik[off]));  // ctor: sug = deg LM (polynomials.cpp:136,144)
    if (r < 0) {
      e.status = (r == -1) ? BB_STATUS_OVERFLOW_PAIRS : (r == -2 ? BB_STATUS_OVERFLOW_BASIS : BB_STATUS_OVERFLOW_EXPONENT);
      return;
    }
    e.nP = (int)(r & 0xffffffffll);
    ct.upp += (unsigned)(r >> 32);
    e.nG++; e.nT += len;
  }
  if (e.nP == 0) e.status = BB_STATUS_DONE;
}

// Full reset of a slot: draws from stream state `rng` when a distribution is set (re-rolling while P comes out
// empty, buchberger.cpp:313-314), else replays staged ideal `fixed_src`.  Out of line (cold): the results go to
// the slot's state record -- (nG, nP, nT, status), rng, rerolls -- and the caller reloads them.
template <int NV>
__device__ __noinline__ void warp_reset_slot(const BBParams& P, int slot, int fixed_src, uint32_t rng,
                                             unsigned long long* ctrow) {
  const int lane = bb_lane();
  Env e;
  e.base = P.arena + (size_t)slot * P.slot_stride;
  e.nG = e.nP = e.nT = 0; e.status = BB_STATUS_EMPTY; e.guard = 0;
  Ctr ct; ct.clear();
  int rerolls = 0;
  if (P.dist.enabled) {
    for (;;) {
      int ok = 1;
      if (P.dist.kind || !gen_binomial_ideal_warp(P, slot, rng)) {
        if (lane == 0) ok = P.dist.kind ? gen_random_ideal(P, slot, rng) : (gen_binomial_ideal(P, slot, rng) ? 1 : 0);
        ok = __shfl_sync(BB_FULL, ok, 0);
        rng = __shfl_sync(BB_FULL, rng, 0);
      }
      __syncwarp();
      if (ok <= 0) { e.nG = e.nP = e.nT = 0; e.status = ok ? BB_STATUS_OVERFLOW_TERMS : BB_STATUS_EMPTY; break; }
      warp_load_ideal<NV>(P, slot, e, ct);
      if (e.status != BB_STATUS_DONE) break;
      rerolls++;
    }
  } else {
    warp_load_ideal<NV>(P, fixed_src, e, ct);
  }
  env_store(P, slot, e);
  if (lane == 0) {
    BBEnvState& S = P.st[slot];
    S.rng = rng; S.rerolls = rerolls;
    S.steps = 0; S.adds = 0; S.zero = 0; S.nonzero = 0; S.truncated = 0;
    S.trace_hash = 0; S.disc_return = 0.0; S.discount = 1.0;
  }
  ct.spill(ctrow);
  __syncwarp();
}

// ---------------------------------------------------------------------------------------------------- hashes
// The per-step checksum of the (i, j, additions) sequence is a rolling polynomial hash mod 2^64,
//   h <- h * 0x9E3779B97F4A7C15 + (i | j << 16 | additions << 32) + 1,
// order-sensitive and one 64-bit multiply-add per step (the position-salted splitmix sum it replaces was 3.7 % of
// k_run's instructions, profiles/README.md v10).  `pair` = (j << 16) | i as the step returns it.  The basis / GB
// checksums below, computed once per episode over many terms in parallel, stay position-salted additive sums.
__device__ __forceinline__ unsigned long long trace_hash_step(unsigned long long h, uint32_t pair, int adds) {
  return h * BB_GOLD + ((((unsigned long long)(uint32_t)adds) << 32) | pair) + 1ull;
}
// lens: polynomial lengths as an int array with the given stride (in ints)
template <int NV>
__device__ __noinline__ unsigned long long warp_terms_hash(const uint64_t* tk, const uint32_t* tc, int nT, const int* lens,
                                                           int lens_stride, int npoly) {
  typedef KL<NV> K;
  const int lane = bb_lane();
  unsigned long long h = 0;
#pragma unroll 1
  for (int t = lane; t < nT; t += 32) {
    const uint64_t k = tk[t];
    uint64_t elo = 0, ehi = 0;
#pragma unroll
    for (int v = 0; v < NV; v++) {
      const uint64_t x = K::exp(k, v);
      if (v < 4) elo |= x << (16 * v); else ehi |= x << (16 * (v - 4));
    }
    h += bb_hash_item_impl((uint64_t)tc[t], 3ull * t) + bb_hash_item_impl(elo, 3ull * t + 1) +
         bb_hash_item_impl(ehi, 3ull * t + 2);
  }
  for (int p = lane; p < npoly; p += 32) h += bb_mix64((uint64_t)lens[(size_t)p * lens_stride] + BB_GOLD2 * (uint64_t)(p + 1));
#pragma unroll
  for (int o = 16; o; o >>= 1) h += bb_shfl64(h, lane ^ o);
  return h;
}

// The same polynomial list (lengths with a stride, as in warp_terms_hash) written to a caller's bb_poly_sink as episode
// `ep`: lane 0 reserves room with two atomics and publishes where[ep] (-1, -1 and used[2] += 1 when it does not fit), the
// lanes unpack the keys into NV int32 exponents.  Once per episode, out of line (cold).
template <int NV>
__device__ __noinline__ void warp_export_polys(const uint64_t* tk, const uint32_t* tc, const int* lens, int lens_stride,
                                               int npoly, int nT, const bb_poly_sink& sink, int ep) {
  typedef KL<NV> K;
  const int lane = bb_lane();
  long long p0 = 0, t0 = 0;
  int ok = 0;
  if (lane == 0) {
    p0 = (long long)atomicAdd(&sink.used_dev[0], (unsigned long long)npoly);
    t0 = (long long)atomicAdd(&sink.used_dev[1], (unsigned long long)nT);
    ok = p0 + npoly <= sink.cap_polys && t0 + nT <= sink.cap_terms;
    if (!ok) atomicAdd(&sink.used_dev[2], 1ull);
    sink.where_dev[2 * (size_t)ep] = ok ? p0 : -1;
    sink.where_dev[2 * (size_t)ep + 1] = ok ? t0 : -1;
  }
  ok = __shfl_sync(BB_FULL, ok, 0);
  if (!ok) return;
  p0 = (long long)bb_shfl64((uint64_t)p0, 0);
  t0 = (long long)bb_shfl64((uint64_t)t0, 0);
  int32_t* lo = sink.lens_dev + p0;
  int32_t* eo = sink.exps_dev + t0 * NV;
  int32_t* co = sink.coefs_dev + t0;
#pragma unroll 1
  for (int p = lane; p < npoly; p += 32) lo[p] = lens[(size_t)p * lens_stride];
#pragma unroll 1
  for (int t = lane; t < nT; t += 32) {
    const uint64_t k = tk[t];
#pragma unroll
    for (int v = 0; v < NV; v++) eo[(size_t)t * NV + v] = (int32_t)K::exp(k, v);
    co[t] = (int32_t)tc[t];
  }
}

// ---------------------------------------------------------------------------------------------------- final GB
// interreduce(minimalize(G)), buchberger.cpp:102-122.  minimalize: G sorted ascending by lead monomial (stable),
// g kept iff no kept lead monomial divides LM g  <=>  no f with LM f strictly dividing LM g and no earlier f
// with the same lead monomial (every lead monomial is divisible by a kept one, by induction along the order).
// interreduce: g <- (1/LC g) * (LT g + reduce(g - LT g, Gmin)), Gmin scanned in ascending-LM order.
// Output goes to the slot's GB arena (gkey/gcoef/glen/gcount).  O(m^2/32) once per episode; reads the slot's state
// record, does not modify the environment.  Returns 1, or 0 on overflow.  Out of line (cold).
template <int NV>
__device__ __noinline__ int warp_final_gb(const BBParams& P, int slot, unsigned long long* ctrow) {
  typedef KL<NV> K;
  const int lane = bb_lane();
  Env e; env_load(P, slot, e);
  Ctr ct; ct.clear();
  const int m = e.nG;
  const uint64_t* lm = ENV_PTR(uint64_t, e, P, o_lm);
  const GHeadMem* gh = ENV_PTR(GHeadMem, e, P, o_ghead);
  uint64_t* gk = P.gkey + (size_t)slot * P.max_terms;
  uint32_t* gc = P.gcoef + (size_t)slot * P.max_terms;
  int* gl = P.glen + (size_t)slot * P.max_basis;
  uint64_t* rlm2 = P.grlm + (size_t)slot * P.max_basis;    // lead monomials of Gmin, ascending
  uint32_t* ridx2 = P.gridx + (size_t)slot * P.max_basis;  // their basis indices
  uint32_t* flag = P.gflag + (size_t)slot * P.max_basis;   // kept flags by basis index
  for (int b0 = 0; b0 < m; b0 += 32) {
    const int g = b0 + lane;
    if (g < m) {
      const uint64_t kg = lm[g];
      bool kept = true;
      for (int o = 0; o < m; o++) {
        const uint64_t ko = lm[o];
        if (ko == kg) kept &= !(o < g);
        else kept &= !K::divides(ko, kg);
      }
      flag[g] = kept ? 1u : 0u;
    }
  }
  __syncwarp();
  int nmin = 0;
  for (int b0 = 0; b0 < m; b0 += 32) {
    const int g = b0 + lane;
    const bool kept = g < m && flag[g] != 0u;
    if (kept) {
      const uint64_t kg = lm[g];
      int rank = 0;  // kept elements with a smaller lead monomial (larger key); kept lead monomials are distinct
      for (int o = 0; o < m; o++) rank += (flag[o] != 0u) && (lm[o] > kg);
      rlm2[rank] = kg; ridx2[rank] = (uint32_t)g;
    }
    nmin += __popc(__ballot_sync(BB_FULL, kept));
  }
  __syncwarp();
  int gT = 0, ok = 1;
  uint64_t* hk = ENV_PTR(uint64_t, e, P, o_hkey);
  uint32_t* hc = ENV_PTR(uint32_t, e, P, o_hcoef);
  const uint64_t* tk = ENV_PTR(uint64_t, e, P, o_tkey);
  const uint32_t* tc = ENV_PTR(uint32_t, e, P, o_tcoef);
  for (int q = 0; q < nmin && ok; q++) {
    const int g = (int)ridx2[q];
    const GHead f = load_head(gh + g);
    if (gT + 1 > P.max_terms) { ok = 0; break; }
    // dividend = g - LT g: copy the tail into scratch half 0
    const int n = (int)f.len - 1;
    if (n > P.max_poly_terms) { ok = 0; break; }
#pragma unroll 1
    for (int t = lane; t < n; t += 32) { hk[t] = tk[f.off + 1 + t]; hc[t] = tc[f.off + 1 + t]; }
    __syncwarp();
    Dividend h;
    h.k0 = h.k1 = 0; h.c0 = h.c1 = 0; h.sug = 0;
    dividend_from_scratch(P, e, h, n, 0);
    int steps;
    const int rlen = warp_reduce<NV>(P, e, h, rlm2, ridx2, nmin, true, gk + gT + 1, gc + gT + 1, P.max_terms - gT - 1, steps,
                                     ct);
    if (rlen < 0) { ok = 0; break; }
    if (lane == 0) { gk[gT] = f.lm; gc[gT] = 1u; gl[q] = 1 + rlen; }
#pragma unroll 1
    for (int t = lane; t < rlen; t += 32) gc[gT + 1 + t] = bbf_mulmod(P.F, gc[gT + 1 + t], f.invlc);
    gT += 1 + rlen;
    __syncwarp();
  }
  if (e.guard & K::g_all) ok = 0;
  if (lane == 0) { P.gcount[2 * slot] = nmin; P.gcount[2 * slot + 1] = gT; }
  ct.spill(ctrow);
  __syncwarp();
  return ok;
}
