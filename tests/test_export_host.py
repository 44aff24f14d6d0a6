"""CPU-side checks of the polynomial export of bb_run_export: the symbol and its struct at the C-ABI, and the canonical
episode order PolyBatch builds from a packed sink (scattered placement, unstored episodes, empty bases)."""
import ctypes as C
import os
import shutil
import subprocess

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_run_export_is_exported():
    from deepgroebner_b200 import _lib
    assert "bb_run_export" in _lib.EXPORTS
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip("libbbenv.so not built (run __graft_entry__.build())")
    lib = _lib.load()
    assert hasattr(C.CDLL(_lib.LIB_PATH), "bb_run_export")
    assert len(lib.bb_run_export.argtypes) == len(lib.bb_run.argtypes) + 2


def test_poly_sink_layout_matches_header(tmp_path):
    from deepgroebner_b200 import _lib
    S = _lib.BBPolySink
    assert C.sizeof(S) == 56
    assert [getattr(S, f).offset for f, _ in S._fields_] == [0, 8, 16, 24, 32, 40, 48]
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler to read the header's layout")
    src = tmp_path / "sink.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "bbenv.h"\nint main(void) {\n'
                   '  printf("%zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(bb_poly_sink), offsetof(bb_poly_sink, lens_dev),\n'
                   '         offsetof(bb_poly_sink, exps_dev), offsetof(bb_poly_sink, coefs_dev), offsetof(bb_poly_sink, where_dev),\n'
                   '         offsetof(bb_poly_sink, used_dev), offsetof(bb_poly_sink, cap_polys), offsetof(bb_poly_sink, cap_terms));\n'
                   '  return 0;\n}\n')
    exe = tmp_path / "sink"
    subprocess.run([cc, "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [C.sizeof(S)] + [getattr(S, f).offset for f, _ in S._fields_]


def packed_sink(episodes, order, nvars=2):
    """A packed sink as the runners leave it: episodes given as lists of polynomials (None = not stored) written in the
    completion order `order`, with a gap of garbage between entries.  Returns the sink tensors and the per-episode sizes
    the records would carry."""
    lens, exps, coefs = [], [], []
    where = torch.full((len(episodes), 2), -1, dtype=torch.int64)
    npolys = torch.zeros(len(episodes), dtype=torch.int32)
    nterms = torch.zeros(len(episodes), dtype=torch.int32)
    for e in order:
        G = episodes[e]
        if G is None:
            npolys[e], nterms[e] = 7, 9      # an unstored episode's record sizes must not matter
            continue
        lens.append(99)
        exps.extend([[-5] * nvars])
        coefs.append(-5)
        where[e, 0], where[e, 1] = len(lens), len(coefs)
        npolys[e], nterms[e] = len(G), sum(len(g) for g in G)
        for g in G:
            lens.append(len(g))
            for c, x in g:
                exps.append(list(x))
                coefs.append(c)
    return (torch.tensor(lens, dtype=torch.int32), torch.tensor(exps, dtype=torch.int32).reshape(-1),
            torch.tensor(coefs, dtype=torch.int32), where, npolys, nterms)


def test_poly_batch_canonical_order_on_cpu():
    from deepgroebner_b200.buchberger import PolyBatch
    eps = [
        [[(1, (2, 0)), (5, (0, 1))], [(1, (0, 3))]],
        None,
        [],
        [[(7, (1, 1))]],
        None,
        [[(1, (4, 0)), (2, (1, 2)), (3, (0, 0))], [(1, (0, 1))], [(9, (0, 0))]],
    ]
    lens, exps, coefs, where, npolys, nterms = packed_sink(eps, order=[5, 3, 1, 0, 2, 4])
    b = PolyBatch.from_sink(lens, exps, coefs, where, npolys, nterms, 2)
    assert len(b) == 6
    assert b.stored.tolist() == [G is not None for G in eps]
    assert b.ep_offsets.tolist() == [0, 2, 2, 2, 3, 3, 6]
    assert b.poly_offsets.tolist() == [0, 2, 3, 4, 7, 8, 9]
    assert b.exps.shape == (9, 2) and b.coefs.tolist() == [1, 5, 1, 7, 1, 2, 3, 1, 9]
    assert [b[e] for e in range(6)] == eps
    assert b.to_lists() == eps
    # another completion order gives the same batch
    b2 = PolyBatch.from_sink(*packed_sink(eps, order=[2, 0, 4, 5, 1, 3]), 2)
    assert b2 == b


def test_poly_batch_of_nothing():
    from deepgroebner_b200.buchberger import PolyBatch
    eps = [None, [], None]
    b = PolyBatch.from_sink(*packed_sink(eps, order=[0, 1, 2], nvars=3), 3)
    assert b.stored.tolist() == [False, True, False]
    assert b.ep_offsets.tolist() == [0, 0, 0, 0] and b.poly_offsets.tolist() == [0]
    assert b.exps.shape == (0, 3) and b.to_lists() == eps
