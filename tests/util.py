"""Shared helpers for the parity tests.

Parity bar (BASELINE.json north_star): integer outputs (anchor selections,
iteration counts, status words) bit-exact; FP64 state and covariance within
1e-9 relative.

The reference algorithm contains discrete decisions taken on floating-point
comparisons (Newton stop test `|cost-newCost|/cost > 1e-3`, the 2-D damping test
`tentativeCost > cost`, the 10000-iteration cap of ML.cpp:67,165, IEKF break
tests, `<=` in the best-group scan).  On some inputs -- mostly exactly-determined
3-D solves (4 rangings, cost -> 0) where the Newton iteration wanders until the
cap -- the REFERENCE'S OWN result changes by up to 1e-3 when an input is moved by
one ulp.  No implementation that differs in rounding (a different LAPACK, FMA
contraction, ...) can reproduce those cases, so they are detected with the oracle
itself and reported separately: a filter/epoch is "stable" when the oracle's
outputs are unchanged (to 1e-10 / exactly for integers) under +-1 ulp
perturbations of its range inputs.  The parity bar applies to every stable unit;
the unstable fraction is asserted to be small and is zero for the 8/16-anchor
BASELINE configurations.
"""
import json
import os

import numpy as np

REL_TOL = 1e-9   # BASELINE.json north_star
STAB_TOL = 1e-10  # oracle-vs-perturbed-oracle agreement that defines "stable"


def _per_unit_float_err(a, b):
    """max over leading axes of |a-b| / max(1, |b|), per unit (last axis)."""
    with np.errstate(invalid="ignore"):
        e = np.abs(a - b) / np.maximum(1.0, np.abs(b))
    e = np.where(np.isnan(a) & np.isnan(b), 0.0, e)
    e = np.where(np.isnan(e), np.inf, e)
    return e.reshape(-1, e.shape[-1]).max(axis=0)


def _per_unit_cov_err(a, b):
    """matrix-norm relative error per unit: max|a-b| / max|b| over the unit's entries."""
    a2 = a.reshape(-1, a.shape[-1]); b2 = b.reshape(-1, b.shape[-1])
    with np.errstate(invalid="ignore", divide="ignore"):
        e = np.abs(a2 - b2).max(axis=0) / np.maximum(np.abs(b2).max(axis=0), 1e-300)
    return np.where(np.isnan(e), np.inf, e)


def unit_errors(got, ref, float_keys=(), cov_keys=(), int_keys=()):
    """Returns (float_err [U], int_mismatch [U] bool)."""
    U = ref[(list(float_keys) + list(cov_keys) + list(int_keys))[0]].shape[-1]
    fe = np.zeros(U)
    im = np.zeros(U, dtype=bool)
    for k in float_keys:
        fe = np.maximum(fe, _per_unit_float_err(np.asarray(got[k]), np.asarray(ref[k])))
    for k in cov_keys:
        fe = np.maximum(fe, _per_unit_cov_err(np.asarray(got[k]), np.asarray(ref[k])))
    for k in int_keys:
        d = np.asarray(got[k]) != np.asarray(ref[k])
        im |= d.reshape(-1, d.shape[-1]).any(axis=0)
    return fe, im


def stable_units(ref, perturbed, float_keys=(), cov_keys=(), int_keys=()):
    """Units whose ORACLE result is insensitive to the +-1 ulp input perturbations."""
    stable = None
    for p in perturbed:
        fe, im = unit_errors(p, ref, float_keys, cov_keys, int_keys)
        s = (fe <= STAB_TOL) & ~im
        stable = s if stable is None else (stable & s)
    return stable


# ---- parity report: every assert_parity call leaves one record (also when it fails); the session
# hook in conftest.py writes them to $KFPOS_PARITY_REPORT when it is set (profiles/parity_rNN.json
# are such reports, committed so that the observed tie counts are on disk).
PARITY_REPORT = []


def _current_test():
    return os.environ.get("PYTEST_CURRENT_TEST", "").split(" ")[0]


def write_parity_report(path):
    if not PARITY_REPORT:
        return
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        json.dump(PARITY_REPORT, f, indent=1)


def assert_parity(got, ref, perturbed, float_keys=(), cov_keys=(), int_keys=(), tol=REL_TOL,
                  min_stable=1.0, max_tie_frac=0.0, tie_tol=1e-3, what="", min_allowed=0):
    """Every stable unit must meet the parity bar; at most `max_tie_frac` of them may instead be
    a rounding-level tie of a discrete decision (error <= tie_tol / an integer flip)."""
    fe, im = unit_errors(got, ref, float_keys, cov_keys, int_keys)
    stable = stable_units(ref, perturbed, float_keys, cov_keys, int_keys) if perturbed else np.ones_like(im)
    frac_stable = stable.mean()
    _ok = (fe <= tol) & ~im
    PARITY_REPORT.append(dict(
        test=_current_test(), what=what, units=int(im.size), stable=int(stable.sum()),
        stable_frac=float(frac_stable), all_units_ok=int(_ok.sum()),
        stable_violations=int((stable & ~_ok).sum()), stable_int_mismatches=int((stable & im).sum()),
        unstable_ok=int((~stable & _ok).sum()),
        worst_stable_float_err=float(fe[stable & ~im].max(initial=0.0)),
        tol=tol, min_stable=min_stable, max_tie_frac=max_tie_frac, tie_tol=float(tie_tol),
        int_keys=list(int_keys), float_keys=list(float_keys) + list(cov_keys)))
    assert frac_stable >= min_stable, f"{what}: only {frac_stable:.4f} of the units are stable in the oracle"
    ok = (fe <= tol) & ~im
    viol = stable & ~ok
    n_viol = int(viol.sum())
    allowed = max(int(min_allowed), int(np.floor(max_tie_frac * stable.sum())))
    worst = float(fe[stable].max()) if stable.any() else 0.0
    assert n_viol <= allowed, (f"{what}: {n_viol} stable units miss the parity bar (allowed {allowed}); "
                               f"worst float err {worst:.3e}, int mismatches {int((im & stable).sum())}")
    if n_viol:
        assert float(fe[viol & ~im].max(initial=0.0)) <= tie_tol, f"{what}: tie error above {tie_tol}"
    return dict(stable=float(frac_stable), worst=worst, ties=n_viol)


def ulp_perturbations(r_m, n_random=4, rel=1e-13, seed=20190816):
    """Perturbed copies of an f64 range tensor that define "stable" (missing rangings, <= 0, untouched):
    +-1 and +-2 ulp on every range, plus `n_random` copies with every range moved by +-rel (random sign
    per element).  rel = 1e-13 is the size of the differences between two correct implementations of
    this arithmetic (re-association, FMA contraction, another LAPACK): a unit whose oracle result
    survives them is one whose result is a property of the algorithm and not of a rounding mode.
    The chaotic selections (4-ranging 3-D subsets) flip under ANY such perturbation with the same
    probability whatever its size (measured: 13 % per perturbation); for those tests n_random is raised
    until one further perturbation flips < 1e-3 of the units that survived (24 is enough, 48 used)."""
    up = np.where(r_m > 0, np.nextafter(r_m, np.inf), r_m)
    dn = np.where(r_m > 0, np.nextafter(r_m, -np.inf), r_m)
    up2 = np.where(r_m > 0, np.nextafter(up, np.inf), r_m)
    dn2 = np.where(r_m > 0, np.nextafter(dn, -np.inf), r_m)
    out = [up, dn, up2, dn2]
    rng = np.random.default_rng(seed)
    for _ in range(n_random):
        sgn = rng.choice([-1.0, 1.0], size=r_m.shape)
        out.append(np.where(r_m > 0, r_m * (1.0 + rel * sgn), r_m))
    return out


def to_metres(r):
    """f64 metres exactly as the library converts the wire formats ((double) mm / 1000)."""
    r = np.asarray(r)
    return r if r.dtype == np.float64 else r.astype(np.float64) / 1000


# kept for simple all-units checks
def rel_err_state(x, ref):
    return float(np.max(_per_unit_float_err(np.asarray(x), np.asarray(ref))))


def rel_err_cov(P, ref):
    return float(np.max(_per_unit_cov_err(np.asarray(P), np.asarray(ref))))
