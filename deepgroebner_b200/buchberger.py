"""Vectorised Buchberger environments on B200: the reference's gym-style API over libbbenv.so.

Mirrors ``deepgroebner.buchberger.BuchbergerEnv`` / ``LeadMonomialsEnv`` (buchberger.py:243-394, 448-542) and the
Cython ``CLeadMonomialsEnv`` (wrapped.pyx:11-38): same constructor keywords, same ``reset()`` / ``step()`` /
``seed()`` contract, same observation matrix, action index and reward semantics -- for ``num_envs`` independent
episodes at once.  With ``num_envs=1`` the return values have the reference's shapes (a ``[len(P), 2nk]`` int32
matrix, a float reward, a bool done).  PyTorch only carries device memory and the CUDA stream; every
environment operation is a hand-written CUDA kernel behind the C-ABI in include/bbenv.h.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from .ideals import BinomialSpec, FixedIdealGenerator, PolySpec, parse_ideal_dist
from .rollout import PairsPolicy

# arena capacities per environment: (max_basis, max_pairs, max_terms, max_poly_terms)
CAPACITY_PRESETS = {
    "binomial": dict(max_basis=512, max_pairs=1024, max_terms=1536, max_poly_terms=64),
    "poly": dict(max_basis=512, max_pairs=2048, max_terms=1 << 14, max_poly_terms=512),
    "general": dict(max_basis=2048, max_pairs=8192, max_terms=1 << 19, max_poly_terms=4096),
}


# default room per episode of the polynomial sinks of run_episodes(return_gb / return_basis), as (polynomials, terms);
# a run that needs more is repeated once with the exact totals.  Measured on the C restatement of the reference (2000
# seeds): reduced bases average 3.6 / 4.0 (3-20-10-weighted) and 17 / 22 (5-5-10-uniform, max 54 / 74) polynomials / terms,
# final bases 63 and 82 terms.  The "poly" and "general" rows are not measured (a fraction of the arena capacities).
SINK_ROOM = {
    "binomial": dict(gb=(24, 32), basis=(64, 128)),
    "poly": dict(gb=(32, 512), basis=(128, 2048)),
    "general": dict(gb=(128, 8192), basis=(512, 32768)),
}
# word index (int32) of the record fields that size an episode's entry in each sink
_REC = {f: np.dtype(_lib.STATS_DTYPE).fields[f][1] // 4 for f in ("nbasis", "nterms", "gb_polys", "gb_terms")}
_SINK_COUNTS = {"gb": ("gb_polys", "gb_terms"), "basis": ("nbasis", "nterms")}


class PolyBatch:
    """Polynomials of every episode of a run, device-resident, in episode order (run_episodes(return_gb / return_basis)).

    ep_offsets int64 [E+1] indexes polynomials, poly_offsets int64 [P+1] indexes terms, exps int32 [T, n], coefs int32 [T]
    in [0, p), stored bool [E] (False: the episode did not end in a state that stores anything).  ``batch[e]`` is the
    ``[(coef, exps), ...]`` list of episode e as final_gb() / basis() return it, or None when nothing was stored."""

    def __init__(self, ep_offsets, poly_offsets, exps, coefs, stored):
        self.ep_offsets, self.poly_offsets, self.exps, self.coefs, self.stored = ep_offsets, poly_offsets, exps, coefs, stored

    def __len__(self):
        return self.stored.numel()

    def to_lists(self):
        """Every episode as batch[e] gives it (one copy to the host)."""
        eo, po = self.ep_offsets.tolist(), self.poly_offsets.tolist()
        ex, cf, st = self.exps.cpu().tolist(), self.coefs.cpu().tolist(), self.stored.tolist()
        out = []
        for e in range(len(st)):
            if not st[e]:
                out.append(None)
                continue
            out.append([[(cf[t], tuple(ex[t])) for t in range(po[q], po[q + 1])] for q in range(eo[e], eo[e + 1])])
        return out

    def __getitem__(self, e):
        e = int(e)
        if not bool(self.stored[e]):
            return None
        q0, q1 = int(self.ep_offsets[e]), int(self.ep_offsets[e + 1])
        po = self.poly_offsets[q0:q1 + 1].tolist()
        ex = self.exps[po[0]:po[-1]].cpu().tolist()
        cf = self.coefs[po[0]:po[-1]].cpu().tolist()
        return [[(cf[t - po[0]], tuple(ex[t - po[0]])) for t in range(po[q], po[q + 1])] for q in range(len(po) - 1)]

    def __eq__(self, other):
        return isinstance(other, PolyBatch) and all(
            torch.equal(getattr(self, f), getattr(other, f)) for f in ("ep_offsets", "poly_offsets", "exps", "coefs", "stored"))

    @staticmethod
    def from_sink(lens, exps, coefs, where, npolys, nterms, nvars):
        """Canonical episode order from a packed bb_poly_sink, with tensor ops on the sink's device: where int64 [E, 2]
        (first polynomial, first term of each episode, -1 where nothing was stored), npolys / nterms [E] the size of each
        episode's entry (taken from the episode records)."""
        dev = where.device
        E = where.shape[0]
        stored = where[:, 0] >= 0
        zero = torch.zeros(1, dtype=torch.int64, device=dev)
        npol = torch.where(stored, npolys.to(torch.int64), 0)
        nter = torch.where(stored, nterms.to(torch.int64), 0)
        ep_offsets = torch.cat([zero, torch.cumsum(npol, 0)])
        term_offsets = torch.cat([zero, torch.cumsum(nter, 0)])
        P, T = (int(x) for x in torch.stack([ep_offsets[-1], term_offsets[-1]]).tolist())
        eps = torch.arange(E, device=dev)
        ep_of_poly = torch.repeat_interleave(eps, npol, output_size=P)
        src_poly = where[ep_of_poly, 0] + torch.arange(P, device=dev) - ep_offsets[ep_of_poly]
        poly_offsets = torch.cat([zero, torch.cumsum(lens[src_poly].to(torch.int64), 0)])
        ep_of_term = torch.repeat_interleave(eps, nter, output_size=T)
        src_term = where[ep_of_term, 1] + torch.arange(T, device=dev) - term_offsets[ep_of_term]
        return PolyBatch(ep_offsets, poly_offsets, exps.view(-1, nvars)[src_term], coefs[src_term], stored)

    @staticmethod
    def from_lists(lists, nvars, device="cuda:0", prime=32003, divisors=False):
        """A batch from host lists: lists[e] is a list of polynomials [(coef, exps), ...], exps of any length whose entries
        beyond nvars are zero.  Terms are sorted descending in grevlex (ascending packed key, the device's order).  Raises
        ValueError on a duplicate monomial, a coefficient outside [1, prime), a negative exponent, and, with
        divisors=True (the lists are divisor lists of reduce()), on the zero polynomial."""
        ep, po, ex, cf = [0], [0], [], []
        for G in lists:
            for f in G:
                terms = []
                for c, e in f:
                    e = tuple(int(x) for x in e)
                    if any(e[nvars:]) or min(e, default=0) < 0:
                        raise ValueError("exponents %r: negative, or a variable beyond nvars=%d" % (e, nvars))
                    e = e[:nvars] + (0,) * (nvars - len(e))
                    if not 0 < int(c) < prime:
                        raise ValueError("coefficient %d is outside [1, %d)" % (int(c), prime))
                    terms.append(((-sum(e),) + e[::-1], int(c), e))   # grevlex: higher degree, then smaller last exponents first
                if divisors and not terms:
                    raise ValueError("the zero polynomial is not a valid divisor")
                terms.sort()
                for a, b in zip(terms, terms[1:]):
                    if a[0] == b[0]:
                        raise ValueError("duplicate monomial %r in a polynomial" % (a[2],))
                ex.extend(t[2] for t in terms)
                cf.extend(t[1] for t in terms)
                po.append(len(cf))
            ep.append(len(po) - 1)
        dev = torch.device(device)
        return PolyBatch(torch.tensor(ep, dtype=torch.int64, device=dev), torch.tensor(po, dtype=torch.int64, device=dev),
                         torch.tensor(ex, dtype=torch.int32).view(-1, nvars).to(dev), torch.tensor(cf, dtype=torch.int32, device=dev),
                         torch.ones(len(lists), dtype=torch.bool, device=dev))


def _group_queries(poly_offsets, exps, coefs, which):
    """The queries of reduce() (polynomial q = terms poly_offsets[q] .. poly_offsets[q + 1] of exps / coefs, reduced by list
    which[q]) reordered so that the queries of one list are adjacent: a stable argsort of which.  Returns (order, offsets,
    exps, coefs, which) of the reordered queries; position i holds query order[i]."""
    dev = which.device
    order = torch.argsort(which, stable=True)
    lens = (poly_offsets[1:] - poly_offsets[:-1])[order]
    offsets = torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), torch.cumsum(lens, 0)])
    T = exps.shape[0]
    src = torch.repeat_interleave(poly_offsets[:-1][order] - offsets[:-1], lens, output_size=T) + torch.arange(T, device=dev)
    return order, offsets, exps[src], coefs[src], which[order]


def _ungroup(order, *grouped):
    """Per-query results of the reordered queries back in input order."""
    out = []
    for t in grouped:
        u = torch.empty_like(t)
        u[order] = t
        out.append(u)
    return out


def _remainder_batch(where, rlen, exps, coefs, ep_offsets, stored, nvars):
    """The remainders in a packed sink (where int64 [Q, 2] and lengths rlen [Q], in query order) as a PolyBatch with the entry
    structure ep_offsets / stored of the dividends: query q is polynomial q, empty where nothing was stored.  An entry counts as
    stored when it was and every one of its queries was."""
    dev = where.device
    Q = where.shape[0]
    ok = where[:, 0] >= 0
    lens = torch.where(ok, rlen.to(torch.int64), 0)
    zero = torch.zeros(1, dtype=torch.int64, device=dev)
    poly_offsets = torch.cat([zero, torch.cumsum(lens, 0)])
    T = int(poly_offsets[-1])
    q_of_term = torch.repeat_interleave(torch.arange(Q, device=dev), lens, output_size=T)
    src = where[q_of_term, 1] + torch.arange(T, device=dev) - poly_offsets[q_of_term]
    E = ep_offsets.numel() - 1
    entry = torch.repeat_interleave(torch.arange(E, device=dev), ep_offsets[1:] - ep_offsets[:-1], output_size=Q)
    missing = torch.zeros(E, dtype=torch.int32, device=dev).index_add_(0, entry, (~ok).to(torch.int32))
    return PolyBatch(ep_offsets, poly_offsets, exps.view(-1, nvars)[src], coefs[src], stored & (missing == 0))


def _nonempty(t):
    """t, or one zero element of its dtype where t is empty (the C-ABI takes no NULL arrays)."""
    return t if t.numel() else torch.zeros(1, dtype=t.dtype, device=t.device)


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def resident_envs(device=0, nvars=3):
    """Slots of one resident wave of bb_run's warp runners: the larger of the general and the two-term runner's waves
    (bb_run launches each with no more warps than its own)."""
    lib = _lib.load()
    n = lib.bb_resident_envs(int(device), int(nvars))
    if n <= 0:
        raise _lib.BBError("bb_resident_envs failed: no CUDA device (no CPU fallback)")
    return n


class BuchbergerEngine:
    """Owns one bb_handle (one GPU).  The two environment classes below are thin views over it."""

    def __init__(self, ideal_dist="3-20-10-uniform", elimination="gebauermoeller", rewards="additions",
                 sort_input=False, sort_reducers=True, k=1, num_envs=1, device="cuda:0", prime=32003,
                 capacity=None, **caps):
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise _lib.BBError("no CUDA device: deepgroebner_b200 has no CPU fallback")
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise ValueError("device must be a CUDA device")
        self._ctor = dict(ideal_dist=ideal_dist, elimination=elimination, rewards=rewards, sort_input=sort_input,
                          sort_reducers=sort_reducers, k=k, device=device, prime=prime, capacity=capacity, **caps)
        self.spec = ideal_dist if isinstance(ideal_dist, (BinomialSpec, PolySpec, FixedIdealGenerator)) \
            else parse_ideal_dist(ideal_dist, prime)
        self.n = self.spec.n if isinstance(self.spec, (BinomialSpec, PolySpec)) else self.spec.nvars()
        self.k, self.num_envs, self.prime = int(k), int(num_envs), int(prime)
        self.elimination, self.rewards = elimination, rewards
        default = {BinomialSpec: "binomial", PolySpec: "poly"}.get(type(self.spec), "general")
        self.preset = capacity or default
        preset = dict(CAPACITY_PRESETS[self.preset])
        gen_caps = {k_: caps.pop(k_) for k_ in ("max_gens", "max_gen_terms") if k_ in caps}
        preset.update(caps)
        if isinstance(self.spec, BinomialSpec):
            max_gens, max_gen_terms = self.spec.s, 2 * self.spec.s
        elif isinstance(self.spec, PolySpec):
            max_gens, max_gen_terms = self.spec.s, self.spec.max_gen_terms()
        else:
            max_gens = len(self.spec.F)
            max_gen_terms = sum(len(f) for f in self.spec.F)
        max_gens = max(max_gens, int(gen_caps.get("max_gens", 0)))   # room for larger ideals staged later (set_ideals)
        max_gen_terms = max(max_gen_terms, int(gen_caps.get("max_gen_terms", 0)))
        cfg = _lib.BBConfig(
            abi_version=_lib.BB_ABI_VERSION, device=self.device.index or 0, nvars=self.n, k=self.k, prime=self.prime,
            elimination=_lib.ELIMINATION[elimination], rewards=_lib.REWARDS[rewards], sort_input=int(sort_input),
            sort_reducers=int(sort_reducers), num_envs=self.num_envs, max_gens=max(max_gens, 1),
            max_gen_terms=max(max_gen_terms, 1), **preset)
        self.caps = preset
        h = C.c_void_p()
        rc = self.lib.bb_create(C.byref(cfg), C.byref(h))
        if rc < 0:
            raise _lib.BBError("bb_create failed (%d): %s" % (rc, self.lib.bb_last_error(None).decode()))
        self.h = h
        self.cols = self.lib.bb_cols(self.h)
        self.sm_count = self.lib.bb_sm_count(self.h)
        if isinstance(self.spec, BinomialSpec):
            s = self.spec
            self._ck(self.lib.bb_set_distribution(self.h, s.d, s.s, _lib.DISTRIBUTION[s.dist], int(s.constants),
                                                  int(s.homogeneous), int(s.pure)), "bb_set_distribution")
        elif isinstance(self.spec, PolySpec):
            s = self.spec
            self._ck(self.lib.bb_set_distribution_poly(self.h, s.d, s.s, float(s.lam), _lib.DISTRIBUTION[s.dist],
                                                       int(s.constants), int(s.homogeneous)), "bb_set_distribution_poly")
        else:
            self.set_ideals([self.spec.F] * self.num_envs)

    def __del__(self):
        h = getattr(self, "h", None)
        if h:
            self.lib.bb_destroy(h)
            self.h = None

    def _ck(self, rc, what):
        return _lib.check(self.lib, self.h, rc, what)

    # ---- inputs
    def seed(self, seed=None):
        """seed(int): environment e gets stream seed + e (num_envs=1: exactly BuchbergerEnv.seed);
        seed(sequence): explicit per-environment seeds."""
        if seed is None:
            return
        self._seed(seed, 0)

    def _seed(self, seed, selection):
        # bb_seed_on: one kernel on the current stream, no allocation, no synchronisation (the reference pattern
        # re-seeds before every episode, randomized_agent.py:141-142)
        with torch.cuda.device(self.device):
            if np.ndim(seed) == 0:
                self._ck(self.lib.bb_seed_on(self.h, None, int(seed), selection, _stream()), "bb_seed_on")
            else:
                a = np.ascontiguousarray(seed, dtype=np.int32)
                assert a.shape == (self.num_envs,)
                self._ck(self.lib.bb_seed_on(self.h, a.ctypes.data_as(C.POINTER(C.c_int32)), 0, selection, _stream()),
                         "bb_seed_on")

    def seed_selection(self, seed=0):
        """Seeds the per-environment stream that 'random' selection draws from (buchberger(..., seed))."""
        self._seed(seed, 1)

    def set_ideals(self, ideals, env_ids=None):
        """ideals: list (one per environment) of lists of polynomials [(coef, exps), ...]."""
        n = self.n
        ideal_off, poly_off, exps, coefs = [0], [0], [], []
        for F in ideals:
            for f in F:
                for c, e in f:
                    e = tuple(e)[:n] + (0,) * max(0, n - len(e))
                    exps.extend(int(x) for x in e)
                    coefs.append(int(c))
                poly_off.append(len(coefs))
            ideal_off.append(len(poly_off) - 1)
        ip = C.POINTER(C.c_int32)
        a_io, a_po = np.asarray(ideal_off, np.int32), np.asarray(poly_off, np.int32)
        a_e, a_c = np.asarray(exps, np.int32), np.asarray(coefs, np.int32)
        ids = None if env_ids is None else np.ascontiguousarray(env_ids, np.int32)
        self._ck(self.lib.bb_set_ideals(self.h, None if ids is None else ids.ctypes.data_as(ip), len(ideals),
                                        a_io.ctypes.data_as(ip), a_po.ctypes.data_as(ip), a_e.ctypes.data_as(ip),
                                        a_c.ctypes.data_as(ip)), "bb_set_ideals")

    # ---- the step path (all device-side, asynchronous on the current torch stream)
    def reset(self, mask=None):
        with torch.cuda.device(self.device):
            if mask is not None:
                mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
            self._ck(self.lib.bb_reset(self.h, _ptr(mask), _stream()), "bb_reset")

    def step(self, actions, reward=None, done=None):
        with torch.cuda.device(self.device):
            actions = torch.as_tensor(actions, device=self.device).to(torch.int32).contiguous().view(-1)
            assert actions.numel() == self.num_envs
            if reward is None:
                reward = torch.empty(self.num_envs, dtype=torch.float64, device=self.device)
            if done is None:
                done = torch.empty(self.num_envs, dtype=torch.uint8, device=self.device)
            self._ck(self.lib.bb_step(self.h, _ptr(actions), _ptr(reward), _ptr(done), _stream()), "bb_step")
        return reward, done

    def step_observe(self, actions, pmax, reward=None, done=None, obs=None, lengths=None):
        """step() and the observation of the new state in ONE launch (bb_step_observe): LeadMonomialsEnv.step as a
        whole.  Returns (obs[N, pmax, cols], lengths[N], reward[N], done[N]) as cuda tensors."""
        with torch.cuda.device(self.device):
            actions = torch.as_tensor(actions, device=self.device).to(torch.int32).contiguous().view(-1)
            assert actions.numel() == self.num_envs
            if reward is None:
                reward = torch.empty(self.num_envs, dtype=torch.float64, device=self.device)
            if done is None:
                done = torch.empty(self.num_envs, dtype=torch.uint8, device=self.device)
            if obs is None:
                obs = torch.empty((self.num_envs, pmax, self.cols), dtype=torch.int32, device=self.device)
            if lengths is None:
                lengths = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
            self._ck(self.lib.bb_step_observe(self.h, _ptr(actions), _ptr(reward), _ptr(done), _ptr(obs), _ptr(lengths),
                                              int(pmax), _stream()), "bb_step_observe")
        return obs, lengths, reward, done

    # ---- the same calls with HOST buffers, as the reference's Cython binding makes them (one launch, one sync each)
    def _host_buffers(self, pmax):
        hb = getattr(self, "_hb", None)
        if hb is None or hb["pmax"] != pmax:
            N = self.num_envs
            hb = dict(pmax=pmax, act=np.zeros(N, np.int32), rew=np.zeros(N, np.float64), done=np.zeros(N, np.uint8),
                      len=np.zeros(N, np.int32), obs=np.full((N, pmax, self.cols), -1, np.int32))
            for k_ in ("act", "rew", "done", "len", "obs"):
                hb["p_" + k_] = C.c_void_p(hb[k_].ctypes.data)
            self._hb = hb
        return hb

    def step_host(self, actions, pmax, pad=True):
        """bb_step_host: actions from host memory; returns numpy views (obs[N, pmax, cols], lengths[N], reward[N],
        done[N]) that the next call overwrites.  pad=False leaves the rows beyond |P| undefined."""
        hb = self._host_buffers(int(pmax))
        hb["act"][...] = actions
        self._ck(self.lib.bb_step_host(self.h, hb["p_act"], hb["p_rew"], hb["p_done"], hb["p_obs"], hb["p_len"],
                                       hb["pmax"], int(pad), _stream()), "bb_step_host")
        return hb["obs"], hb["len"], hb["rew"], hb["done"]

    def reset_host(self, pmax, pad=True):
        """bb_reset_host: reset() of every environment and the first observation, to host memory."""
        hb = self._host_buffers(int(pmax))
        self._ck(self.lib.bb_reset_host(self.h, hb["p_obs"], hb["p_len"], hb["pmax"], int(pad), _stream()), "bb_reset_host")
        return hb["obs"], hb["len"]

    def observe_host(self, pmax, pad=True):
        hb = self._host_buffers(int(pmax))
        self._ck(self.lib.bb_observe_host(self.h, hb["p_obs"], hb["p_len"], hb["pmax"], int(pad), _stream()), "bb_observe_host")
        return hb["obs"], hb["len"]

    def select(self, strategy="degree", out=None):
        with torch.cuda.device(self.device):
            if out is None:
                out = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
            self._ck(self.lib.bb_select(self.h, _lib.SELECTION[strategy], _ptr(out), _stream()), "bb_select")
        return out

    def lengths(self):
        with torch.cuda.device(self.device):
            out = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
            self._ck(self.lib.bb_observe(self.h, None, _ptr(out), 0, _stream()), "bb_observe")
        return out

    def observe(self, pmax, obs=None, lengths=None):
        with torch.cuda.device(self.device):
            if obs is None:
                obs = torch.empty((self.num_envs, pmax, self.cols), dtype=torch.int32, device=self.device)
            if lengths is None:
                lengths = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
            self._ck(self.lib.bb_observe(self.h, _ptr(obs), _ptr(lengths), int(pmax), _stream()), "bb_observe")
        return obs, lengths

    def pairs(self, pmax):
        with torch.cuda.device(self.device):
            out = torch.empty((self.num_envs, pmax, 2), dtype=torch.int32, device=self.device)
            lengths = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
            self._ck(self.lib.bb_pairs(self.h, _ptr(out), _ptr(lengths), int(pmax), _stream()), "bb_pairs")
        return out, lengths

    def status(self):
        with torch.cuda.device(self.device):
            out = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
            self._ck(self.lib.bb_status(self.h, _ptr(out), _stream()), "bb_status")
        return out

    def stats(self):
        """Running per-environment episode records as a numpy structured array (synchronises)."""
        with torch.cuda.device(self.device):
            buf = torch.empty(self.num_envs * C.sizeof(_lib.BBEpisodeStats), dtype=torch.uint8, device=self.device)
            self._ck(self.lib.bb_stats(self.h, _ptr(buf), _stream()), "bb_stats")
            return buf.cpu().numpy().view(np.dtype(_lib.STATS_DTYPE))

    # ---- batch management (SURVEY north_star: finished / diverged episodes are compacted)
    def compact(self, out=None):
        """int32 cuda tensor [N + 1]: the number of RUNNING environments, then every slot with the RUNNING ones first
        (bb_compact).  step() / step_observe() do this themselves when auto-reset is off."""
        with torch.cuda.device(self.device):
            if out is None:
                out = torch.empty(self.num_envs + 1, dtype=torch.int32, device=self.device)
            self._ck(self.lib.bb_compact(self.h, _ptr(out), _stream()), "bb_compact")
        return out

    def set_prefetch(self, depth=8):
        """Queues of prepared next episodes per environment for reset() / auto-reset (bb_set_prefetch); 0 = off.  The default
        is 8 for engines of at least 64 environments.  What an environment draws does not change."""
        self._ck(self.lib.bb_set_prefetch(self.h, int(depth)), "bb_set_prefetch")

    def set_serve(self, on=True):
        """One-environment engines answer step_host / reset_host / observe_host through a resident warp polling a mailbox in
        mapped host memory (bb_set_serve; the default for num_envs == 1); off: one kernel launch per call."""
        self._ck(self.lib.bb_set_serve(self.h, int(bool(on))), "bb_set_serve")

    def set_compaction(self, on=True):
        self._ck(self.lib.bb_set_compaction(self.h, int(bool(on))), "bb_set_compaction")

    def status_summary(self):
        """{status name: number of environments} (bb_status_summary; synchronises).  'diverged' sums the faults."""
        counts = np.zeros(_lib.STATUS_COUNT, np.int32)
        with torch.cuda.device(self.device):
            self._ck(self.lib.bb_status_summary(self.h, counts.ctypes.data_as(C.POINTER(C.c_int32)), _stream()),
                     "bb_status_summary")
        out = {_lib.STATUS_NAMES[i]: int(counts[i]) for i in range(_lib.STATUS_COUNT)}
        out["diverged"] = int(counts[3:9].sum())
        return out

    def set_max_episode_length(self, max_steps=0):
        """Episodes of step() / rollout() are cut once they have MORE than max_steps steps (pg.py:470-471); 0 = never."""
        self._ck(self.lib.bb_set_max_episode_length(self.h, int(max_steps or 0)), "bb_set_max_episode_length")

    def set_obs_nvars(self, n_obs):
        """State matrices show the first n_obs variables only (bb_set_obs_nvars: the C++ FixedIdealGenerator quirk)."""
        self._ck(self.lib.bb_set_obs_nvars(self.h, int(n_obs)), "bb_set_obs_nvars")
        self.cols = self.lib.bb_cols(self.h)

    # ---- whole episodes
    def prepare_episodes(self, episodes=None, seed_base=0, seeds=None):
        """The preparation half of the NEXT run_episodes call (bb_prepare) on the current stream -- call it under
        `torch.cuda.stream(side)` to overlap it with a runner at work on another stream.  `seeds`: None for
        seed_base + e, an int32 cuda tensor, or an int32 HOST tensor (pinned: copied asynchronously into one of three
        device buffers of the engine, on the current stream).  Returns the device seeds tensor (or None): pass THAT
        object as `seeds` to the run_episodes call this preparation is for."""
        episodes = self.num_envs if episodes is None else int(episodes)
        with torch.cuda.device(self.device):
            if seeds is not None:
                assert torch.is_tensor(seeds) and seeds.dtype == torch.int32 and seeds.numel() == episodes
                if not seeds.is_cuda:
                    ring = getattr(self, "_seed_ring", None)
                    if ring is None or ring[0].numel() != episodes:
                        ring = self._seed_ring = [torch.empty(episodes, dtype=torch.int32, device=self.device) for _ in range(3)]
                        self._seed_turn = 0
                    dev = ring[self._seed_turn]
                    self._seed_turn = (self._seed_turn + 1) % 3
                    dev.copy_(seeds, non_blocking=True)
                    seeds = dev
            self._ck(self.lib.bb_prepare(self.h, episodes, int(seed_base), _ptr(seeds), _stream()), "bb_prepare")
        return seeds

    def set_episode_offset(self, offset=0):
        """Global index of episode 0 of the following run_episodes calls (bb_set_episode_offset; sharding.py)."""
        self._ck(self.lib.bb_set_episode_offset(self.h, int(offset)), "bb_set_episode_offset")

    def set_timing(self, on=True):
        self._ck(self.lib.bb_set_timing(self.h, int(bool(on))), "bb_set_timing")

    def last_run_ms(self):
        """(preparation ms, runner ms) of the last run_episodes call (first batch); needs set_timing(True)."""
        a, b = C.c_float(0), C.c_float(0)
        self._ck(self.lib.bb_last_run_ms(self.h, C.byref(a), C.byref(b)), "bb_last_run_ms")
        return float(a.value), float(b.value)

    def run_episodes(self, strategy="degree", episodes=None, seed_base=0, seeds=None, max_steps=0, gamma=0.99,
                     compute_gb=False, trace_episodes=0, trace_cap=0, to_host=True, selection_seed=0, out_host=None,
                     out=None, return_gb=False, return_basis=False, gb_capacity=None, basis_capacity=None, greedy=False,
                     policy_counter=0):
        """Runs `episodes` episodes to completion with on-device selection (bb_run_export).  Returns (stats, trace):
        stats is a structured array of bb_episode_stats (numpy if to_host else a uint8 cuda tensor), trace an
        int32 [trace_episodes, trace_cap, 4] array of (i, j, additions, |P| after), -1 padded.
        seeds: per-episode ideal-stream seeds, a numpy array or an int32 torch tensor (pinned host memory is copied
        asynchronously); out_host: a pinned uint8 host tensor of episodes * 72 bytes that receives the records (the
        returned array is a view of it); out: a uint8 cuda tensor of episodes * 72 bytes for the records instead of the
        engine's own buffer (calls in flight on different streams need different ones).
        return_gb / return_basis: also return every episode's reduced Groebner basis (return_gb implies compute_gb; stored
        for episodes that end done) and / or final basis G in insertion order (episodes that end done or are cut by
        max_steps), as (stats, trace, {"gb": PolyBatch, "basis": PolyBatch}).  gb_capacity / basis_capacity: room of each
        sink as (polynomials, terms) over the whole call (default: SINK_ROOM per episode of the capacity preset).  A run
        whose polynomials do not fit is repeated once with the exact totals -- a second run of the same episodes, with
        the same records (runs are deterministic).  Reading the sinks' fill synchronises the stream.
        strategy may also be a rollout.PairsPolicy built for this engine's cols: its head chooses every pair (bb_run_policy),
        sampling (greedy=False) or taking the argmax, lowest row on ties (greedy=True).  Step t of episode e of the call
        draws its uniform from stream net.seed + (episode offset + e) and counter policy_counter + t, so environment e of
        the step API seeded seed_base + e and stepped with policy(net, counter=policy_counter + t) plays the same episode;
        selection_seed does not apply."""
        episodes = self.num_envs if episodes is None else int(episodes)
        want = [k for k, on in (("gb", return_gb), ("basis", return_basis)) if on]
        compute_gb = compute_gb or return_gb
        net = strategy if isinstance(strategy, PairsPolicy) else None
        with torch.cuda.device(self.device):
            if net is not None:
                W = net.device_weights(self.device, self.cols)
            nbytes = max(episodes, 1) * C.sizeof(_lib.BBEpisodeStats)
            buf = out if out is not None else getattr(self, "_run_buf", None)
            if out is not None:
                assert out.is_cuda and out.dtype == torch.uint8 and out.numel() >= nbytes
            elif buf is None or buf.numel() < nbytes:
                buf = self._run_buf = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            trace = None
            if trace_episodes > 0 and trace_cap > 0:
                trace = torch.full((trace_episodes, trace_cap, 4), -1, dtype=torch.int32, device=self.device)
            d_seeds = None
            if seeds is not None:
                if torch.is_tensor(seeds) and seeds.is_cuda:
                    assert seeds.dtype == torch.int32 and seeds.numel() == episodes
                    d_seeds = seeds
                elif torch.is_tensor(seeds):
                    assert seeds.dtype == torch.int32 and seeds.numel() == episodes
                    d_seeds = getattr(self, "_run_seeds", None)
                    if d_seeds is None or d_seeds.numel() != episodes:
                        d_seeds = self._run_seeds = torch.empty(episodes, dtype=torch.int32, device=self.device)
                    d_seeds.copy_(seeds, non_blocking=True)
                else:
                    d_seeds = torch.as_tensor(np.ascontiguousarray(seeds, np.int32), device=self.device)
                    assert d_seeds.numel() == episodes
            room = {"gb": gb_capacity, "basis": basis_capacity}
            for k in want:
                if room[k] is None:
                    room[k] = tuple(episodes * x for x in SINK_ROOM[self.preset][k])
            for attempt in range(2):
                sinks = {k: self._sink(episodes, *room[k]) for k in want}
                tail = (int(max_steps), float(gamma), int(bool(compute_gb)), _ptr(buf), _ptr(trace), int(trace_episodes),
                        int(trace_cap), _stream(), sinks["gb"][1] if "gb" in sinks else None,
                        sinks["basis"][1] if "basis" in sinks else None)
                if net is not None:
                    self._ck(self.lib.bb_run_policy(self.h, net.hidden, *[_ptr(t) for t in W], int(net.seed),
                                                    int(policy_counter), int(bool(greedy)), episodes, int(seed_base),
                                                    _ptr(d_seeds), *tail), "bb_run_policy")
                else:
                    self._ck(self.lib.bb_run_export(self.h, _lib.SELECTION[strategy], episodes, int(seed_base), _ptr(d_seeds),
                                                    int(selection_seed), *tail), "bb_run_export")
                if not want:
                    break
                used = {k: sinks[k][0]["used"].tolist() for k in want}
                if attempt or all(used[k][2] == 0 for k in want):
                    break
                room = {k: (used[k][0], used[k][1]) for k in want}
            polys = {}
            if want:
                rec = buf[:episodes * C.sizeof(_lib.BBEpisodeStats)].view(torch.int32).view(-1, C.sizeof(_lib.BBEpisodeStats) // 4)
                for k in want:
                    t = sinks[k][0]
                    fp, ft = _SINK_COUNTS[k]
                    polys[k] = PolyBatch.from_sink(t["lens"], t["exps"], t["coefs"], t["where"], rec[:, _REC[fp]],
                                                   rec[:, _REC[ft]], self.n)
            if not to_host:
                return (buf[:nbytes], trace, polys) if want else (buf[:nbytes], trace)
            if out_host is not None:
                out_host[:nbytes].copy_(buf[:nbytes], non_blocking=True)
                torch.cuda.current_stream().synchronize()
                stats = out_host.numpy().view(np.dtype(_lib.STATS_DTYPE))[:episodes]
            else:
                stats = buf[:nbytes].cpu().numpy().view(np.dtype(_lib.STATS_DTYPE))[:episodes]
            trace = trace.cpu().numpy() if trace is not None else None
            return (stats, trace, polys) if want else (stats, trace)

    def _sink(self, episodes, polys, terms):
        """Device buffers of one bb_poly_sink for `episodes` episodes and its ctypes struct."""
        d, i32 = self.device, torch.int32
        t = dict(lens=torch.empty(max(int(polys), 1), dtype=i32, device=d),
                 exps=torch.empty(max(int(terms), 1) * self.n, dtype=i32, device=d),
                 coefs=torch.empty(max(int(terms), 1), dtype=i32, device=d),
                 where=torch.empty((max(episodes, 1), 2), dtype=torch.int64, device=d)[:episodes],
                 used=torch.zeros(3, dtype=torch.int64, device=d))
        s = _lib.BBPolySink(lens_dev=t["lens"].data_ptr(), exps_dev=t["exps"].data_ptr(), coefs_dev=t["coefs"].data_ptr(),
                            where_dev=t["where"].data_ptr(), used_dev=t["used"].data_ptr(), cap_polys=int(polys),
                            cap_terms=int(terms))
        return t, C.byref(s), s

    def reduce(self, polys, divisors, which=None, sorted=False, return_remainders=True, capacity=None):
        """reduce(g, F) (buchberger.cpp:24-49) on the device (bb_reduce): every polynomial of entry e of the PolyBatch `polys`
        is reduced by the polynomials of entry which[e] of the PolyBatch `divisors` (default: entry e), e.g. a run_episodes
        (return_gb=True) batch, passed as it is.  sorted=False scans each list in its order; True scans it stable-sorted by
        ascending lead monomial (the order of a reduced basis from run_episodes, where both give the same remainders).
        Queries are grouped by list on the device; results come back in input order.  Returns (remainders, steps, lengths,
        status): remainders a PolyBatch with the entry structure of `polys` (None with return_remainders=False, which attaches
        no sink), steps / lengths / status int32 cuda tensors per polynomial (status 2 = done, BB_STATUS_* or -1 for
        malformed input; a query that is not done has an empty remainder, and its entry is not stored).  A divisor entry
        that was not stored gives its queries status -1.  capacity: the remainders' sink room as (polynomials, terms); a
        call whose remainders do not fit is repeated once with the exact totals (a second launch, which the counters count).
        Like run_episodes, a call on the stream of the step API overwrites its environments."""
        dev, n = self.device, self.n
        i32, i64 = torch.int32, torch.int64
        with torch.cuda.device(dev):
            if polys.exps.shape[1] != n or divisors.exps.shape[1] != n:
                raise ValueError("both batches need %d exponents per term" % n)
            E, L = len(polys), len(divisors)
            ep = polys.ep_offsets.to(dev)
            Q = polys.poly_offsets.numel() - 1
            w = torch.arange(E, device=dev) if which is None else torch.as_tensor(which, device=dev).to(i64).view(-1)
            if w.numel() != E:
                raise ValueError("which needs one list per entry of polys")
            if L:
                ok = (w >= 0) & (w < L) & divisors.stored.to(dev)[w.clamp(0, L - 1)]
                w = torch.where(ok, w, -1)
            else:
                w = torch.full_like(w, -1)
            which_q = torch.repeat_interleave(w, ep[1:] - ep[:-1], output_size=Q).to(i32)
            order, q_off, q_ex, q_cf, wq = _group_queries(polys.poly_offsets.to(dev), polys.exps.to(dev), polys.coefs.to(dev),
                                                          which_q)
            steps, rlen, status = (torch.zeros(Q, dtype=i32, device=dev) for _ in range(3))
            d = [t.to(dev).contiguous() for t in (divisors.ep_offsets, divisors.poly_offsets, divisors.exps, divisors.coefs)]
            args = [L] + [_nonempty(t) for t in d] + [Q, q_off, _nonempty(q_ex.contiguous()), _nonempty(q_cf), wq]
            room = capacity or (Q, max(2 * int(q_ex.shape[0]), 1024))
            sink = None
            for attempt in range(2 if Q else 0):
                sink = self._sink(Q, *room) if return_remainders else None
                self._ck(self.lib.bb_reduce(self.h, *[a if isinstance(a, int) else _ptr(a) for a in args], int(bool(sorted)),
                                            _ptr(steps), _ptr(rlen), _ptr(status), sink[1] if sink else None, _stream()),
                         "bb_reduce")
                if sink is None:
                    break
                used = sink[0]["used"].tolist()
                if attempt or used[2] == 0:
                    break
                room = (used[0], used[1])
            steps, rlen, status = _ungroup(order, steps, rlen, status)
            rem = None
            if return_remainders:
                where = _ungroup(order, sink[0]["where"])[0] if sink else torch.full((Q, 2), -1, dtype=i64, device=dev)
                t = sink[0] if sink else dict(exps=torch.zeros(0, dtype=i32, device=dev), coefs=torch.zeros(0, dtype=i32, device=dev))
                rem = _remainder_batch(where, rlen, t["exps"], t["coefs"], ep, polys.stored.to(dev), n)
        return rem, steps, rlen, status

    def value(self, strategy="degree", gamma=0.99, rollouts=None, selection_seed=0, max_steps=0, out=None):
        """BuchbergerEnv.value for every environment (bb_value): float64 cuda tensor [N].  strategy is a selection
        name or 'sample' (1 Degree + 100 Random rollouts, best kept, buchberger.cpp:333-341).  rollouts: None = the
        reference's count (101 for 'sample', 1 otherwise); for 'sample' it includes the Degree rollout."""
        code = _lib.VALUE_SAMPLE if strategy == "sample" else _lib.SELECTION[strategy]
        if rollouts is None:
            rollouts = 0 if strategy == "sample" else 1   # bb_value: 0 -> 101 for BB_VALUE_SAMPLE
        with torch.cuda.device(self.device):
            if out is None:
                out = torch.empty(self.num_envs, dtype=torch.float64, device=self.device)
            self._ck(self.lib.bb_value(self.h, code, float(gamma), int(rollouts), int(selection_seed), int(max_steps),
                                       _ptr(out), _stream()), "bb_value")
        return out

    def set_auto_reset(self, on=True):
        """Finished environments are reset inside step() / rollout() (vector-env semantics, bb_set_auto_reset)."""
        self._ck(self.lib.bb_set_auto_reset(self.h, int(bool(on))), "bb_set_auto_reset")

    def set_wide(self, mode=-1):
        """How run_episodes reduces (bb_set_wide): -1 auto, 0 materialised dividend, 1 dividend as a set of streams run by
        one CTA per environment (long polynomials); 2 / 3 as 1 with 6 / 48 stream slots (consolidation path), 7 as 1 with
        8 register slots (shared-memory table), 8 as 1 with 32 reducers in the control warp's registers (memory scan of the
        rest); 4 / 5 / 6 are kept for compatibility and equal 1 / 2 / 3.  Results are identical; only speed differs."""
        self._ck(self.lib.bb_set_wide(self.h, int(mode)), "bb_set_wide")

    def set_prepare_mode(self, by_warp=False):
        """Episode preparation of run_episodes (bb_set_prepare_mode): one thread per episode where it applies
        (default) or always one warp per episode.  Results are identical; only speed differs."""
        self._ck(self.lib.bb_set_prepare_mode(self.h, int(bool(by_warp))), "bb_set_prepare_mode")

    def set_two_term(self, on=True):
        """Runner of run_episodes for binomial distributions (bb_set_two_term): True (default) the two-term runner, False the
        general one.  Both give bit-identical results; the switch exists to compare them."""
        self._ck(self.lib.bb_set_two_term(self.h, int(bool(on))), "bb_set_two_term")

    def set_selection_seed_stride(self, stride=1):
        """run_episodes seeds episode e's 'random' selection stream with selection_seed + e * stride
        (0: one seed for every episode, as scripts/make_strat.cpp does)."""
        self._ck(self.lib.bb_set_selection_seed_stride(self.h, int(stride)), "bb_set_selection_seed_stride")

    def policy(self, net, counter=0, greedy=False, return_all=False, pmax=None):
        """PMLP head + categorical sample on the current states (bb_policy_pmlp).  net: rollout.PairsPolicy.
        Returns (actions int32 [N], logprob float32 [N][, logprobs float32 [N, pmax] padded with -inf])."""
        with torch.cuda.device(self.device):
            W1, b1, w2, b2 = net.device_weights(self.device, self.cols)
            actions = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
            logp = torch.empty(self.num_envs, dtype=torch.float32, device=self.device)
            allp = None
            if return_all:
                pmax = int(pmax or self.caps["max_pairs"])
                allp = torch.full((self.num_envs, pmax), float("-inf"), dtype=torch.float32, device=self.device)
            self._ck(self.lib.bb_policy_pmlp(self.h, net.hidden, _ptr(W1), _ptr(b1), _ptr(w2), _ptr(b2), int(net.seed),
                                             int(counter), int(bool(greedy)), _ptr(actions), _ptr(logp), _ptr(allp),
                                             int(pmax or 0), _stream()), "bb_policy_pmlp")
        return (actions, logp, allp) if return_all else (actions, logp)

    def rollout(self, net, T, counter0=0, greedy=False, store_obs=False, pmax=None, out=None):
        """T fused steps of every environment (bb_rollout).  Returns a dict of [N, T] cuda tensors: actions, logp,
        reward, done, lengths (+ obs [N, T, pmax, cols] when store_obs)."""
        N, dev = self.num_envs, self.device
        with torch.cuda.device(dev):
            W1, b1, w2, b2 = net.device_weights(dev, self.cols)
            o = out or {}
            o.setdefault("actions", torch.empty((N, T), dtype=torch.int32, device=dev))
            o.setdefault("logp", torch.empty((N, T), dtype=torch.float32, device=dev))
            o.setdefault("reward", torch.empty((N, T), dtype=torch.float32, device=dev))
            o.setdefault("done", torch.empty((N, T), dtype=torch.uint8, device=dev))
            o.setdefault("lengths", torch.empty((N, T), dtype=torch.int32, device=dev))
            obs = None
            if store_obs:
                pmax = int(pmax or 64)
                obs = o.setdefault("obs", torch.empty((N, T, pmax, self.cols), dtype=torch.int32, device=dev))
            self._ck(self.lib.bb_rollout(self.h, net.hidden, _ptr(W1), _ptr(b1), _ptr(w2), _ptr(b2), int(net.seed),
                                         int(counter0), int(bool(greedy)), int(T), _ptr(o["actions"]), _ptr(o["logp"]),
                                         _ptr(o["reward"]), _ptr(o["done"]), _ptr(o["lengths"]), _ptr(obs),
                                         int(pmax or 0), _stream()), "bb_rollout")
        return o

    def copy_env(self, dst_env, src, src_env):
        """Environment src_env of engine `src` -> environment dst_env of this engine (bb_copy_env)."""
        with torch.cuda.device(self.device):
            self._ck(self.lib.bb_copy_env(self.h, int(dst_env), src.h, int(src_env), _stream()), "bb_copy_env")

    def clone(self):
        """A new engine with the same configuration and a copy of every environment (the copy constructor)."""
        other = BuchbergerEngine(num_envs=self.num_envs, **self._ctor)
        for e in range(self.num_envs):
            other.copy_env(e, self, e)
        return other

    # ---- host views
    def _polys_out(self, fn, env, what):
        cap_p, cap_t = self.caps["max_basis"], self.caps["max_terms"]
        lens = np.zeros(cap_p, np.int32)
        exps = np.zeros(cap_t * self.n, np.int32)
        coefs = np.zeros(cap_t, np.int32)
        nt = C.c_int(0)
        ip = C.POINTER(C.c_int32)
        with torch.cuda.device(self.device):
            torch.cuda.current_stream().synchronize()
            np_ = self._ck(fn(self.h, int(env), lens.ctypes.data_as(ip), cap_p, exps.ctypes.data_as(ip),
                              coefs.ctypes.data_as(ip), cap_t, C.byref(nt)), what)
        out, t = [], 0
        E = exps.reshape(-1, self.n)
        for q in range(np_):
            out.append([(int(coefs[t + r]), tuple(int(x) for x in E[t + r])) for r in range(lens[q])])
            t += int(lens[q])
        return out

    def basis(self, env=0):
        """G of one environment in insertion order: [[(coef, exps), ...], ...] (BuchbergerEnv.G)."""
        return self._polys_out(self.lib.bb_download_basis, env, "bb_download_basis")

    def final_gb(self, env=0):
        """interreduce(minimalize(G)) computed on device (buchberger.cpp:102-122, 265)."""
        return self._polys_out(self.lib.bb_final_gb, env, "bb_final_gb")

    def counters(self, reset=False):
        c = _lib.BBCounters()
        self._ck(self.lib.bb_counters_read(self.h, C.byref(c), int(reset)), "bb_counters_read")
        return c.as_dict()


class LeadMonomialsEnv:
    """A BuchbergerEnv whose state is the matrix of the pairs' lead monomials (buchberger.py:448-542).

    Extra keywords over the reference: ``num_envs`` (N independent episodes), ``device``, ``pmax`` (row capacity
    of the batched observation; default max_pairs).  Returns for N == 1 match the reference exactly; for N > 1:
    ``reset() -> (obs[N, pmax, 2nk] int32 padded with -1, lengths[N])``,
    ``step(actions[N]) -> ((obs, lengths), reward[N] float64, done[N] bool, {})``.
    """

    def __init__(self, ideal_dist="3-20-10-uniform", elimination="gebauermoeller", rewards="additions",
                 sort_input=False, sort_reducers=True, k=1, dtype=np.int32, num_envs=1, device="cuda:0", pmax=None,
                 compat_cxx_nvars=False, max_episode_length=None, **engine_kwargs):
        self.engine = BuchbergerEngine(ideal_dist, elimination, rewards, sort_input, sort_reducers, k, num_envs,
                                       device, **engine_kwargs)
        if compat_cxx_nvars and isinstance(self.engine.spec, FixedIdealGenerator):
            # the C++ / Cython env shows max(variable index in use) variables for a fixed ideal (ideals.cpp:146-154)
            used = [v for f in self.engine.spec.F for _, e in f for v, x in enumerate(e) if x]
            self.engine.set_obs_nvars(max(1, max(used) if used else 1))
        if max_episode_length:
            self.engine.set_max_episode_length(max_episode_length)
        self.k, self.dtype, self.num_envs = k, dtype, num_envs
        self.pmax = int(pmax) if pmax else self.engine.caps["max_pairs"]

    def seed(self, seed=None):
        self.engine.seed(seed)

    def _state(self):
        if self.num_envs == 1:
            obs, lengths = self.engine.observe_host(self.pmax, pad=False)
            return obs[0, :int(lengths[0])].astype(self.dtype)
        return self.engine.observe(self.pmax)

    def reset(self):
        if self.num_envs == 1:   # one launch pair, one synchronisation (wrapped.pyx:18-21)
            obs, lengths = self.engine.reset_host(self.pmax, pad=False)
            return obs[0, :int(lengths[0])].astype(self.dtype)
        self.engine.reset()
        return self._state()

    def step(self, action):
        if self.num_envs == 1:   # one launch, one synchronisation, the action in the launch parameters (wrapped.pyx:23-26)
            obs, lengths, reward, done = self.engine.step_host(action, self.pmax, pad=False)
            return obs[0, :int(lengths[0])].astype(self.dtype), float(reward[0]), bool(done[0]), {}
        obs, lengths, reward, done = self.engine.step_observe(action, self.pmax)
        return (obs, lengths), reward, done.bool(), {}

    def value(self, strategy="degree", gamma=0.99, **kw):
        """Discounted return of finishing from the current state under `strategy` (wrapped.pyx:32-33,
        buchberger.cpp:332-351); a float for num_envs == 1, else a float64 cuda tensor [N]."""
        v = self.engine.value(strategy, gamma, **kw)
        return float(v.item()) if self.num_envs == 1 else v

    def copy(self):
        """Deep copy including the ideal stream (wrapped.pyx:35-38)."""
        other = object.__new__(type(self))
        other.__dict__.update(self.__dict__)
        other.engine = self.engine.clone()
        return other


class BuchbergerEnv:
    """Buchberger's algorithm as an environment (buchberger.py:243-394): state (G, P), action a pair (i, j).

    For N == 1 ``reset()`` returns ``(G, P)`` with G a list of polynomials ``[(coef, exps), ...]`` (downloaded
    from the device) and P a list of pairs; for N > 1 the state is ``(pairs[N, pmax, 2], lengths[N])`` and G is
    available per environment through ``basis(env)``.  Coefficients are those of the reference's C++ env (basis
    elements are not made monic, SURVEY quirk Q3)."""

    def __init__(self, ideal_dist="3-20-10-uniform", elimination="gebauermoeller", rewards="additions",
                 sort_input=False, sort_reducers=True, num_envs=1, device="cuda:0", pmax=None, **engine_kwargs):
        self.engine = BuchbergerEngine(ideal_dist, elimination, rewards, sort_input, sort_reducers, 1, num_envs,
                                       device, **engine_kwargs)
        self.num_envs = num_envs
        self.pmax = int(pmax) if pmax else self.engine.caps["max_pairs"]

    def seed(self, seed=None):
        self.engine.seed(seed)

    def basis(self, env=0):
        return self.engine.basis(env)

    def value(self, strategy="degree", gamma=0.99, **kw):
        """buchberger.py:380-387 / buchberger.cpp:332-351."""
        v = self.engine.value(strategy, gamma, **kw)
        return float(v.item()) if self.num_envs == 1 else v

    def copy(self):
        other = object.__new__(type(self))
        other.__dict__.update(self.__dict__)
        other.engine = self.engine.clone()
        return other

    def _state(self):
        if self.num_envs == 1:
            n = int(self.engine.lengths().item())
            pairs, _ = self.engine.pairs(max(n, 1))
            P = [tuple(int(x) for x in row) for row in pairs[0, :n].cpu().numpy()]
            return self.engine.basis(0), P
        return self.engine.pairs(self.pmax)

    def reset(self):
        self.engine.reset()
        return self._state()

    def step(self, action):
        """action: a pair (i, j) (N == 1) or an int tensor [N, 2]."""
        pairs, lengths = self.engine.pairs(self.pmax)
        a = torch.as_tensor(action, device=pairs.device).to(torch.int32).view(self.num_envs, 1, 2)
        hit = (pairs == a).all(-1)
        rows = torch.where(hit.any(1), hit.int().argmax(1), torch.full_like(lengths, -1)).to(torch.int32)
        if self.num_envs == 1 and int(rows.item()) < 0:
            raise ValueError("pair %r is not in the pair set" % (tuple(action),))
        reward, done = self.engine.step(rows)
        state = self._state()
        if self.num_envs == 1:
            return state, float(reward.item()), bool(done.item()), {}
        return state, reward, done.bool(), {}


class BuchbergerAgent:
    """Built-in selection strategies computed on device (buchberger.py:397-439, buchberger.cpp:160-241):
    first, degree, normal, sugar, random, last, codegree, strange, spice."""

    def __init__(self, selection="normal"):
        self.strategy = selection

    def act(self, env):
        """LeadMonomialsEnv: row indices [N] (an int for num_envs == 1); BuchbergerEnv: pairs [N, 2] (a tuple (i, j)
        for num_envs == 1), as buchberger.py:397-439 returns them."""
        rows = env.engine.select(self.strategy)
        if isinstance(env, BuchbergerEnv):
            pairs, _ = env.engine.pairs(env.pmax)
            picked = pairs[torch.arange(env.num_envs, device=pairs.device), rows.long().clamp(0, env.pmax - 1)]
            return tuple(int(x) for x in picked[0].cpu()) if env.num_envs == 1 else picked
        return int(rows.item()) if env.num_envs == 1 else rows
