"""Vectorised float64 restatement of the BCD phase search (`optimize_phase_shift`, MARL/Environment.py:208-231)
that also reports how close each decision was.

The reference objective of env e is `sum_v K_v |S|^2` with `S = sum_m theta_m c_m`,
`c_m = sum_v phases_R_i[v, m] * phase_R[m]` and `K_v > 0` independent of theta (EnvOracle._objective), so the
search is the same as one on |S|^2: for each element m in order, every candidate phase e_k is scored as
`|S - theta_m c_m + e_k c_m|^2`, the first maximum wins and it is accepted only if it is > 0 (the reference starts
from `best = 0` and tests `best < x`); otherwise theta_m becomes the integer 0.  All envs and candidates are scored
at once, one element at a time.

`margin` is `(best - runner_up) / best` of each decision.  Where it is small, a few ulps of difference in how the
objective is evaluated can change the choice; above a threshold the choice is determined by the geometry alone.
"""
import cmath

import numpy as np


def candidates(control_bit):
    """The reference's candidate phasors, evaluated as it does (MARL/Environment.py:169,213)."""
    angles = np.linspace(0, 2 * np.pi, 2 ** int(control_bit), endpoint=False)
    return np.array([cmath.exp(ph * 1j) for ph in angles])


def coefficients(oracle):
    """c[e, m] = sum_v phases_R_i[e, v, m] * phase_R[m] of an `EnvOracle` after `compute_parms`."""
    return oracle.phases_R_i.sum(axis=1) * oracle.phase_R[None, :]


def bcd_search(c, theta0, control_bit, n=None):
    """Run the BCD search from `theta0` [E, M] on the coefficients `c` [E, M].

    `n` [E] (optional): env e searches its first n[e] elements only (a per-env RIS size); its elements m >= n[e]
    keep their theta and stay out of S.  Returns `(theta, index, margin)`: theta [E, M] complex; index [E, M] int,
    the chosen candidate, -1 where nothing was accepted (theta = 0) and -2 where the element is not searched;
    margin [E, M] float, 1 where there is a single candidate, 0 where nothing was accepted, NaN where not searched."""
    c = np.asarray(c, dtype=complex)
    theta = np.array(theta0, dtype=complex, copy=True)
    E, M = c.shape
    n = np.full(E, M) if n is None else np.asarray(n).reshape(E)
    cand = candidates(control_bit)
    active = np.arange(M)[None, :] < n[:, None]
    S = np.sum(np.where(active, theta * c, 0), axis=1)
    index = np.full((E, M), -2, dtype=np.int64)
    margin = np.full((E, M), np.nan)
    for m in range(M):
        on = active[:, m]
        if not on.any():
            break
        rest = S - theta[:, m] * c[:, m]
        z = rest[:, None] + cand[None, :] * c[:, m, None]
        val = z.real * z.real + z.imag * z.imag
        k = np.argmax(val, axis=1)  # the first maximum
        best = val[np.arange(E), k]
        ok = best > 0.0
        if len(cand) > 1:
            runner = np.partition(val, -2, axis=1)[:, -2]
            mg = np.where(ok, (best - runner) / np.where(ok, best, 1.0), 0.0)
        else:
            mg = np.where(ok, 1.0, 0.0)
        new = np.where(ok, cand[k], 0.0)
        theta[:, m] = np.where(on, new, theta[:, m])
        S = np.where(on, rest + new * c[:, m], S)
        index[:, m] = np.where(on, np.where(ok, k, -1), -2)
        margin[:, m] = np.where(on, mg, np.nan)
    return theta, index, margin


def choice_index(theta, control_bit, tol):
    """The candidate index of each theta [E, M] (-1 for theta = 0).  Raises unless every theta is 0 or within `tol`
    of a candidate: |theta * conj(e_k) - 1| <= tol."""
    theta = np.asarray(theta, dtype=complex)
    nc = 2 ** int(control_bit)
    cand = candidates(control_bit)
    zero = theta == 0
    k = np.rint(np.angle(theta) / (2 * np.pi / nc)).astype(np.int64) % nc
    err = np.where(zero, 0.0, np.abs(theta * np.conj(cand[k]) - 1.0))
    if not (err <= tol).all():
        i = tuple(np.argwhere(~(err <= tol))[0])
        raise AssertionError(f"theta{i} = {theta[i]!r} is not a candidate phasor within {tol:g} (off by {err[i]:.3g})")
    return np.where(zero, -1, k)


def compare_choices(got, want, margin, control_bit, free0, threshold):
    """Compare chosen indices `got` with the reference's `want` and its `margin` (both from `bcd_search` /
    `choice_index`; elements with want == -2 are not compared).

    An env is excluded when one of its decisions has margin < `threshold`.  `free0` (bool, or [E] bool) marks the
    envs whose element 0 is searched while every other element is out of S: a start from theta = 0, or a single
    element.  There S - theta_0 c_0 = 0, so every candidate scores |c_0|^2, an exact tie in exact arithmetic that
    rounding breaks at random.  It is not a decision: whichever candidate wins, the rest of the search is the same
    up to that rotation, so the env's indices are compared after shifting them by the difference at element 0.
    Returns (excluded [E] bool, wrong [E] bool); `wrong` is False on excluded envs."""
    got, want = np.asarray(got), np.asarray(want)
    nc = 2 ** int(control_bit)
    free0 = np.broadcast_to(np.asarray(free0, dtype=bool), (len(want),))
    decided = want != -2
    decided[:, 0] &= ~free0
    excluded = (decided & (margin < threshold)).any(axis=1)
    shift = np.where(free0 & (got[:, 0] >= 0) & (want[:, 0] >= 0), got[:, 0] - want[:, 0], 0) % nc
    expect = np.where(want >= 0, (want + shift[:, None]) % nc, want)
    wrong = ((got != expect) & (want != -2)).any(axis=1) & ~excluded
    return excluded, wrong
