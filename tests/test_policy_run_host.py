"""CPU checks of the policy runner's public surface: the exported symbol and its prototype, and the refusals of the
list-level calls that happen before any device work."""
import pytest


def test_symbol_declared_and_bound():
    import os
    from deepgroebner_b200 import _lib
    assert "bb_run_policy" in _lib.EXPORTS
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "bbenv.h")).read()
    assert "int bb_run_policy(bb_handle* h, int hidden," in hdr


def test_policy_columns_must_fit_the_ideals():
    """Ideals in 3 variables have 6 k state columns: a 10-column policy is refused before an engine is built, and a name
    that is not a strategy is refused as before."""
    from deepgroebner_b200.rollout import PairsPolicy
    from deepgroebner_b200.strat import groebner_bases, parse_ideal_string, strategy_stats
    ideals = [parse_ideal_string("b-a^2|c-a^3")]
    with pytest.raises(ValueError, match="10 state columns"):
        strategy_stats(ideals, PairsPolicy(10, hidden=32))
    with pytest.raises(ValueError, match="state columns"):
        groebner_bases(ideals, selection=PairsPolicy(4, hidden=32))
    with pytest.raises(ValueError, match="unknown strategy"):
        strategy_stats(ideals, "best")
