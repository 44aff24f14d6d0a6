"""deepgroebner_b200 -- B200-native (sm_100a) batched Buchberger environment.

Drop-in for the environment path of dylanpeifer/deepgroebner (BuchbergerEnv / LeadMonomialsEnv reset/step),
vectorised over N episodes per GPU.  The CUDA library (libbbenv.so, C-ABI in include/bbenv.h) is required:
there is no CPU fallback.  Importing this package does not load CUDA; constructing an environment does.
"""
from .ideals import BinomialSpec, FixedIdealGenerator, PolySpec, cyclic, parse_ideal_dist  # noqa: F401

__all__ = ["BuchbergerEnv", "LeadMonomialsEnv", "BuchbergerEngine", "BuchbergerAgent", "BinomialSpec", "PolySpec",
           "FixedIdealGenerator", "cyclic", "parse_ideal_dist", "groebner_bases",
           "reduce_polynomials"]


def __getattr__(name):  # torch / CUDA are only pulled in when an environment class is requested
    if name in ("BuchbergerEnv", "LeadMonomialsEnv", "BuchbergerEngine", "BuchbergerAgent"):
        from . import buchberger
        return getattr(buchberger, name)
    if name in ("groebner_bases", "reduce_polynomials"):
        from . import strat
        return getattr(strat, name)
    raise AttributeError(name)
