"""The vectorised BCD search of `oracle/bcd_oracle.py` against the oracle's own `optimize_phase_shift`, the direct
restatement of the reference loop: every phase resolution the library accepts up to 64 candidates, V and M from
1 to 70, and the three kinds of start the drivers produce (all-zero arena, off-grid phases of `get_next_phase`,
grid phases of `Random_phase`)."""
import numpy as np
import pytest

from oracle.bcd_oracle import bcd_search, candidates, choice_index, coefficients, compare_choices
from oracle.env_oracle import EnvOracle

# (control_bit, V, M): every control_bit 0..6, every V of {1, 3, 8, 9} and every M of {1, 7, 40, 70}
CASES = [(0, 8, 40), (0, 1, 7), (1, 3, 40), (1, 9, 1), (2, 8, 7), (2, 1, 70), (3, 9, 40), (3, 3, 70), (4, 8, 70),
         (4, 3, 7), (5, 1, 40), (5, 9, 7), (6, 8, 40), (6, 3, 1)]
STARTS = ("zero", "offgrid", "grid")
E = 16
# Both sides evaluate the same objective in float64, in a different order (the reference sums V * M products per
# candidate, the restatement updates S); at M <= 70 their margins differ by ~1e-15, far below this threshold (the
# one tests/test_gpu_bcd.py uses against the kernels).
THRESHOLD = 1e-12


def geometry(E, V, M, control_bit, seed):
    rng = np.random.default_rng(seed)
    o = EnvOracle("marl", V, M, control_bit, E=E)
    o.set_vehicles(rng.uniform(0, 400, (E, V, 2)), np.zeros((E, V), int), np.full((E, V), 10))
    o.compute_parms()
    return o, rng


def start(o, kind, rng):
    if kind == "offgrid":
        o.get_next_phase(rng.uniform(0, 2 * np.pi, (o.E, o.M)))
    elif kind == "grid":
        o.random_phase(rng.integers(0, 2 ** o.control_bit, (o.E, o.M)))


@pytest.mark.parametrize("control_bit,V,M", CASES)
def test_bcd_search_matches_oracle(control_bit, V, M):
    for kind in STARTS:
        o, rng = geometry(E, V, M, control_bit, 1000 * control_bit + 10 * V + M)
        start(o, kind, rng)
        theta, idx, margin = bcd_search(coefficients(o), o.elements_phase_shift_complex, control_bit)
        o.optimize_phase_shift()
        want = o.elements_phase_shift_complex
        cand = candidates(control_bit)
        ref_idx = choice_index(want, control_bit, 1e-15)
        assert np.array_equal(np.where(ref_idx >= 0, cand[ref_idx], 0), want)  # the candidate values themselves
        excluded, wrong = compare_choices(idx, ref_idx, margin, control_bit, kind == "zero" or M == 1, THRESHOLD)
        assert not wrong.any(), f"{kind}: envs {np.flatnonzero(wrong)} chose differently"
        assert excluded.sum() == 0, f"{kind}: {excluded.sum()} envs with a decision margin < {THRESHOLD:g}"
        if kind != "zero" and M > 1:
            assert np.array_equal(theta, want)


def test_bcd_search_per_env_size():
    """A per-env RIS size n[e] searches the first n[e] elements exactly as a handle with M = n[e] would, and keeps
    the rest."""
    control_bit, V, M = 3, 8, 40
    o, rng = geometry(E, V, M, control_bit, 7)
    start(o, "offgrid", rng)
    n = rng.integers(1, M + 1, E)
    n[0], n[1] = 1, M
    theta0 = o.elements_phase_shift_complex.copy()
    theta, idx, margin = bcd_search(coefficients(o), theta0, control_bit, n)
    c = coefficients(o)
    for e in range(E):
        th_e, idx_e, mg_e = bcd_search(c[e:e + 1, :n[e]], theta0[e:e + 1, :n[e]], control_bit)
        assert np.array_equal(theta[e, :n[e]], th_e[0]) and np.array_equal(idx[e, :n[e]], idx_e[0])
        np.testing.assert_allclose(margin[e, :n[e]], mg_e[0], rtol=1e-9)
        assert np.array_equal(theta[e, n[e]:], theta0[e, n[e]:]) and (idx[e, n[e]:] == -2).all()


def test_bcd_search_tie_and_zero_rules():
    """Exact ties go to the smallest index; a search whose every candidate scores 0 stores theta = 0."""
    c = np.array([[1.0, 0.0, 1.0j], [0.0, 0.0, 0.0]])
    theta0 = np.array([[1.0, 1.0j, 1.0], [0.0, 0.0, 0.0]], dtype=complex)
    theta, idx, margin = bcd_search(c, theta0, 2)
    assert idx[0, 1] == 0 and theta[0, 1] == 1.0 and margin[0, 1] == 0.0  # c_1 = 0: every candidate ties
    assert (idx[1] == -1).all() and (theta[1] == 0).all() and (margin[1] == 0).all()
