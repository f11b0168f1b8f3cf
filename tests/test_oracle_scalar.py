"""Config 1 (real scalar Laplace geometric MG): the numpy oracle against the reference's own golden iteration
counts (NB/2c_analysis_mass_variation_non-telescoping.ipynb:555-598, reproduced by the S2 binary) and against
the S2 binary itself when oracle/_ref/s2_mgrid is present."""
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

from oracle import scalar_s2 as S

GOLDEN_3LVL = {0.02: 448, 0.04: 114, 0.08: 29, 0.10: 19, 0.14: 10, 0.17: 8, 0.20: 7}   # NB/2c...:587-593
GOLDEN_4LVL = {0.02: 113, 0.04: 29, 0.08: 9, 0.10: 9, 0.20: 7}                           # NB/2c...:594-598
GOLDEN_2LVL = {0.06: 205, 0.08: 116, 0.10: 75, 0.14: 39, 0.17: 27, 0.20: 20}             # NB/2c...:555-562 (ntl_1copy rows)


@pytest.mark.parametrize("nlevels,table", [(3, GOLDEN_3LVL), (4, GOLDEN_4LVL), (2, GOLDEN_2LVL)])
def test_golden_iteration_counts(nlevels, table):
    for m, want in table.items():
        if want > 250:
            continue   # keep the CPU suite short; the 448-iteration row is covered by test_vs_s2_binary
        got, _, _ = S.solve(64, m, nlevels, 3, 0)
        assert got == want, (nlevels, m, got, want)


def _s2_binary(repo_root):
    path = os.path.join(repo_root, "oracle", "_ref", "s2_mgrid")      # built by `make -C oracle REF=<reference source tree>`
    return path if os.path.exists(path) else None


@pytest.mark.parametrize("args", [(32, 0.1, 1, 3, 0), (32, 0.2, 2, 20, 0), (64, 0.02, 3, 3, 0), (64, 0.1, 3, 3, 1),
                                  (32, 0.1, 0, 5, 0), (16, 0.3, 2, 2, 1)])
def test_vs_s2_binary(repo_root, args):
    exe = _s2_binary(repo_root)
    if exe is None:
        pytest.skip("oracle/_ref/s2_mgrid not built (make -C oracle REF=<reference source tree>)")
    L, m, nl, ni, tf = args
    with tempfile.TemporaryDirectory() as d:
        out = subprocess.run([exe, str(L), str(m), str(nl), str(ni), str(tf)], cwd=d, capture_output=True, text=True).stdout
        ans = int(re.search(r"Ans (\d+)", out).group(1))
        last = open(os.path.join(d, "results_phi.txt")).read().strip().split("\n")[-1].rstrip(",").split(",")
        phi_ref = np.array([float(v) for v in last[1:]]).reshape(L, L).T.reshape(-1)   # file is x outer, y inner
    got, phi, _ = S.solve(L, m, nl, ni, tf)
    assert got == ans
    assert np.max(np.abs(phi - phi_ref)) < 2e-6   # the file keeps 6 decimals (%f)


def test_edge_cases():
    with pytest.raises(ValueError):
        S.solve(8, 0.1, 3, 3)            # max_levels = log2(L)-1 (S2:218)
    it, phi, hist = S.solve(8, 0.5, 2, 3)
    assert it >= 0 and hist[-1] < 1e-13


# "Loop breaks at iteration N" as printed by the S1 binaries that oracle/Makefile builds (targets _ref/s1_mgrid_L*)
S1_BINARY_ITERS = {(32, 0.1, 2, 3): 231, (32, 0.05, 3, 20): 31}


@pytest.mark.parametrize("L,m,nl,ni", [(32, 0.1, 2, 3), (32, 0.05, 3, 20)])
def test_s1_variant_vs_binary(L, m, nl, ni):
    """BASELINE configs[0] literally: code/1_laplace_scalar/2D_laplace_Mgrid.cpp (hard-coded constants patched at
    build time by oracle/Makefile) against oracle.scalar_s2.solve_s1, through the iteration count the binary printed."""
    got, _, hist = S.solve_s1(L, m, nl, ni)
    assert got == S1_BINARY_ITERS[(L, m, nl, ni)]
