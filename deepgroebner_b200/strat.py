"""Strategy statistics over a file of ideals: the contract of the reference's scripts/make_strat.cpp, one launch.

The reference reads ``data/stats/<dist>/<dist>.csv`` (a header line, then one ideal per line as polynomials separated
by ``|``, e.g. ``a^2*b+c*d|b^3-7*a``; written by scripts/make_dist.m2:62-72), runs ``buchberger(F, strategy,
GebauerMoeller, Additions, false, true, 0.99, seed)`` on every line (make_strat.cpp:64-70) and writes
``data/stats/<dist>/<dist>_<strategy>[_<seed>].csv`` with the columns ``ZeroReductions,NonzeroReductions,
PolynomialAdditions``.  Here every ideal of the file is staged on the device (bb_set_ideals) and all of them run to
completion in one bb_run launch; the output file is byte-identical to the reference binary's.  groebner_bases runs the
same staging and returns what buchberger() returns first: the reduced Groebner basis of every ideal of the list.
"""
import os

STRATEGIES = ("first", "degree", "normal", "sugar", "random", "last", "codegree", "strange", "spice")
HEADER = "ZeroReductions,NonzeroReductions,PolynomialAdditions"
NVARS_MAX = 8  # polynomials.h:29


def parse_polynomial(s, prime=32003):
    """parse_polynomial (polynomials.cpp:226-300): variables a..h, ``^`` powers, ``*`` products, integer
    coefficients, ``+``/``-`` between terms, no spaces.  Returns [(coef in [1,p), exponent 8-tuple)] in the order
    written, equal monomials summed (Polynomial operator+, polynomials.cpp:148-177) and zero sums dropped."""
    i, n = 0, len(s)

    def monomial():
        nonlocal i
        e = [0] * NVARS_MAX
        while True:
            if i >= n:
                return e
            v = ord(s[i]) - ord("a")
            if v < 0 or v >= NVARS_MAX:
                raise ValueError("invalid variable name %r in %r" % (s[i], s))
            i += 1
            power = 1
            if i < n and s[i] == "^":
                i += 1
                j = i
                while j < n and s[j].isdigit():
                    j += 1
                if j == i:
                    raise ValueError("missing exponent in %r" % s)
                power, i = int(s[i:j]), j
            e[v] += power
            if i < n and s[i] == "*":
                i += 1
                continue
            return e

    terms = {}
    order = []
    while i < n:
        sign = 1
        while i < n and s[i] in "+-":
            if s[i] == "-":
                sign = -sign
            i += 1
        if i < n and s[i].isdigit():
            j = i
            while j < n and s[j].isdigit():
                j += 1
            c, i = int(s[i:j]), j
            if i < n and s[i] == "*":
                i += 1
                e = monomial()
            else:
                e = [0] * NVARS_MAX
        else:
            c, e = 1, monomial()
        e = tuple(e)
        if e not in terms:
            order.append(e)
            terms[e] = 0
        terms[e] = (terms[e] + sign * c) % prime
    return [(terms[e], e) for e in order if terms[e]]


def parse_ideal_string(line, prime=32003):
    """parse_ideal_string (make_strat.cpp:12-19): polynomials separated by '|'."""
    return [parse_polynomial(p, prime) for p in line.split("|")]


def read_ideal_file(path, prime=32003):
    with open(path) as fh:
        lines = fh.read().split("\n")
    if lines and lines[-1] == "":
        lines.pop()
    return [parse_ideal_string(line, prime) for line in lines[1:]]  # the first line is the column name


def _policy(selection):
    """The rollout.PairsPolicy that `selection` is, else None after checking that it names a built-in strategy."""
    from .rollout import PairsPolicy
    if isinstance(selection, PairsPolicy):
        return selection
    if selection not in STRATEGIES:
        raise ValueError("unknown strategy %r" % selection)
    return None


def _staged_engine(ideals, device, capacity, caps, policy=None, **env_kw):
    """An engine with one environment per ideal of the list, each ideal staged on the device (bb_set_ideals), and every
    episode's Random-selection stream seeded with the same seed (make_strat.cpp:66).  With a PairsPolicy the engine's k
    is the one whose state matrices have the policy's columns: net.cols = 2 n k for ideals in n variables."""
    from .buchberger import BuchbergerEngine
    from .ideals import FixedIdealGenerator
    n = 1
    for F in ideals:
        for f in F:
            if not f:
                raise ValueError("the zero polynomial is not a valid generator")
            for _, e in f:
                for v, x in enumerate(e):
                    if x:
                        n = max(n, v + 1)
    if policy is not None:
        k = policy.cols // (2 * n)
        if k < 1 or 2 * n * k != policy.cols:
            raise ValueError("the policy has %d state columns, but ideals in %d variables have 2 * %d * k for k = 1, 2, ..."
                             % (policy.cols, n, n))
        env_kw["k"] = k
    binomial = all(len(f) <= 2 for F in ideals for f in F)
    eng = BuchbergerEngine(FixedIdealGenerator(ideals[0], n), num_envs=len(ideals), device=device,
                           capacity=capacity or ("binomial" if binomial else "poly"),
                           max_gens=max(len(F) for F in ideals),
                           max_gen_terms=max(sum(len(f) for f in F) for F in ideals), **env_kw, **caps)
    eng.set_ideals(ideals)
    eng.set_selection_seed_stride(0)
    return eng


CAPACITY_ADVICE = "raise the arena capacities (capacity='general' or max_basis/max_pairs/max_terms keywords)"


def _check_finished(stats):
    bad = (stats["status"] != 2).nonzero()[0]
    if len(bad):
        raise RuntimeError("ideal %d did not finish (status %d): %s" % (int(bad[0]), int(stats["status"][bad[0]]),
                                                                         CAPACITY_ADVICE))


def strategy_stats(ideals, strategy, seed=0, device="cuda:0", capacity=None, greedy=False, **caps):
    """(zero_reductions, nonzero_reductions, polynomial_additions) int arrays for a list of ideals: one bb_run launch
    with every ideal staged on the device.  `seed`: the Random-selection seed shared by every ideal
    (make_strat.cpp:66 passes the same optional seed to every buchberger() call).  `strategy` may be a
    rollout.PairsPolicy (bb_run_policy): ideal i is episode i, whose step t samples with stream strategy.seed + i and
    counter t (greedy=True: the argmax); `seed` does not apply."""
    net = _policy(strategy)
    eng = _staged_engine(ideals, device, capacity, caps, policy=net)
    stats, _ = eng.run_episodes(strategy, episodes=len(ideals), selection_seed=int(seed or 0), gamma=0.99, greedy=greedy)
    _check_finished(stats)
    return stats["zero_reductions"], stats["nonzero_reductions"], stats["additions"]


def groebner_bases(ideals, selection="degree", elimination="gebauermoeller", sort_reducers=True, seed=0, prime=32003,
                   device="cuda:0", capacity=None, greedy=False, **caps):
    """buchberger(F, selection, elimination, Additions, false, sort_reducers, 0.99, seed) (buchberger.cpp:125-266) for
    every ideal of a list in one launch.  Returns (bases, stats): bases[i] is the reduced Groebner basis of ideals[i]
    (interreduce(minimalize(G)), ascending lead monomial, monic) in the form parse_ideal_string gives -- a list of
    [(coef, 8 exponents), ...] -- and stats the episode records (bb_episode_stats).  write_ideal_file(path, bases)
    writes them in the file notation.  An ideal that does not finish raises, as in strategy_stats.  `selection` may be a
    rollout.PairsPolicy, sampled or (greedy=True) argmax, as in strategy_stats; the reduced bases do not depend on it."""
    net = _policy(selection)
    eng = _staged_engine(ideals, device, capacity, caps, policy=net, elimination=elimination, sort_reducers=sort_reducers,
                         prime=prime)
    stats, _, out = eng.run_episodes(selection, episodes=len(ideals), selection_seed=int(seed or 0), gamma=0.99,
                                     return_gb=True, greedy=greedy)
    _check_finished(stats)
    pad = (0,) * (NVARS_MAX - eng.n)
    bases = [[[(c, e + pad) for c, e in g] for g in G] for G in out["gb"].to_lists()]
    return bases, stats


def reduce_polynomials(polys, divisors, sorted=False, prime=32003, device="cuda:0", capacity=None, **caps):
    """reduce(g, F) (buchberger.cpp:24-49) for lists of polynomials, on the device in one launch: polys[i] is a list of
    polynomials, each reduced by the list divisors[i], all in the form parse_ideal_string gives ([(coef, exponents), ...]).
    sorted=False scans each divisor list in its order, True stable-sorted by ascending lead monomial.  Returns (remainders,
    steps): remainders[i][j] is the remainder of polys[i][j] ([(coef, 8 exponents), ...], descending grevlex, not made monic)
    and steps[i][j] its number of reduction steps.
    When divisors[i] is a Groebner basis of an ideal I (groebner_bases gives reduced ones), the remainder of g is its normal
    form modulo I, and it is empty exactly when g lies in I.  A reduction that overflows the arena capacities raises."""
    from .buchberger import BuchbergerEngine, PolyBatch, resident_envs
    from .ideals import FixedIdealGenerator
    import torch
    if len(polys) != len(divisors):
        raise ValueError("one divisor list per list of polynomials")
    n = 1
    for L in (polys, divisors):
        for F in L:
            for f in F:
                for _, e in f:
                    for v, x in enumerate(e):
                        if x:
                            n = max(n, v + 1)
    P = PolyBatch.from_lists(polys, n, device, prime=prime)
    D = PolyBatch.from_lists(divisors, n, device, prime=prime, divisors=True)
    envs = max(1, min(len(divisors), resident_envs(torch.device(device).index or 0, n)))
    eng = BuchbergerEngine(FixedIdealGenerator([[(1, (0,) * n)]], n), num_envs=envs, device=device, prime=prime,
                           capacity=capacity or "poly", **caps)
    rem, steps, _, status = eng.reduce(P, D, sorted=sorted)
    st = status.cpu().numpy()
    bad = (st != 2).nonzero()[0]
    if len(bad):
        raise RuntimeError("polynomial %d of the call did not reduce (status %d): %s" % (int(bad[0]), int(st[bad[0]]),
                                                                                      CAPACITY_ADVICE))
    pad = (0,) * (NVARS_MAX - n)
    ep, sp = P.ep_offsets.tolist(), steps.tolist()
    remainders = [[[(c, e + pad) for c, e in r] for r in R] for R in rem.to_lists()]
    return remainders, [sp[ep[i]:ep[i + 1]] for i in range(len(polys))]


def make_strat(dist, strategy, seed=None, root="data/stats", device="cuda:0", **caps):
    """scripts/make_strat.cpp main(): same input/output file names, same refusal to overwrite, same CSV bytes.
    Returns (exit code, message): 0 ok, 2 no distribution file, 3 output exists (make_strat.cpp:35-48)."""
    in_name = os.path.join(root, dist, dist + ".csv")
    if not os.path.exists(in_name):
        return 2, "No distribution file found. Run scripts/make_dist.m2 first."
    out_name = os.path.join(root, dist, "%s_%s.csv" % (dist, strategy))
    if seed is not None and strategy == "random":
        out_name = os.path.join(root, dist, "%s_%s_%s.csv" % (dist, strategy, seed))
    if os.path.exists(out_name):
        return 3, "Output file %s already exists. Delete or move it first." % out_name
    if strategy == "random" and seed is None:
        raise ValueError("random selection needs a seed here (the reference falls back to std::random_device)")
    ideals = read_ideal_file(in_name)
    rows = []
    if ideals:
        z, nz, adds = strategy_stats(ideals, strategy, seed=seed, device=device, **caps)
        rows = ["%d,%d,%d" % (int(a), int(b), int(c)) for a, b, c in zip(z, nz, adds)]
    with open(out_name, "w") as fh:
        fh.write("\n".join([HEADER] + rows) + "\n")
    return 0, out_name


def format_polynomial(f, prime=32003):
    """A polynomial [(coef, exps), ...] in the file's notation (what Macaulay2's toString prints and
    parse_polynomial reads back): ``413*a^2*b^5*c+32*d^2-5``; coefficients above p/2 are written negative."""
    out = []
    for c, e in f:
        c = int(c) % prime
        if c > prime // 2:
            c -= prime
        mono = "*".join(("%s^%d" % (chr(97 + v), x) if x > 1 else chr(97 + v)) for v, x in enumerate(e) if x)
        if not mono:
            body = str(abs(c))
        elif abs(c) == 1:
            body = mono
        else:
            body = "%d*%s" % (abs(c), mono)
        out.append(("-" if c < 0 else ("+" if out else "")) + body)
    return "".join(out) if out else "0"


def write_ideal_file(path, ideals, prime=32003):
    """data/stats/<dist>/<dist>.csv as scripts/make_dist.m2:52-72 writes it: 'Ideal', then one ideal per line."""
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with open(path, "w") as fh:
        fh.write("Ideal\n")
        for F in ideals:
            fh.write("|".join(format_polynomial(f, prime) for f in F) + "\n")
