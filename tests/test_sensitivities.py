"""Solution sensitivities (reference: d_ocp_qp_ipm_sens_frw / _adj behind the plugin's eval_forw_sens / eval_adj_sens,
external/hpipm/ocp_qp/x_ocp_qp_ipm.c:3285-3444): one substitution with the factorisation of the last IPM iteration.

CPU part: the oracle's restatement against the unmodified reference, through its outputs stored by
tests/golden/make_reference_outputs.py (a seeded sample of each sensitivity field with an entry in every stage, and the
field's max |.|).  GPU part: the CUDA path (cuipm_sens_host, through the C ABI) against the oracle.

Tolerances.  The sensitivities are evaluated at the last IPM iterate, where the slacks t of active constraints are
1e-9..1e-16: an absolute difference of 1e-12 between two solvers' iterates (what the solve parity test allows) is a
relative difference of up to 1e-2 in Gamma = lam / t of weakly active constraints, and the linearised KKT system moves
with it.  So: instances on which the two SOLUTIONS agree to round-off (lam and t elementwise to 1e-13 relative; the
majority) must agree in dux / dpi / dt to 1e-9 relative, the others to 1e-2.  dlam (and the adjoint
dt = dt / t) of active constraints are lam/t * (a difference of O(1) numbers that cancels to ~1e-11): the reference's own
value carries ~1e-3 relative error there, those arrays are held to 2e-2 throughout."""
import os

import numpy as np
import pytest

from acados_b200.binding import default_opts
from test_oracle_vs_reference import CASES, GOLD, input_fingerprint, ref_decode, reference_outputs

SENS_CASES = ["c1_mass_spring", "c2_chain_mass", "rand_box", "rand_general", "rand_soft", "rand_masked", "rand_x0_free", "unconstrained"]


def _seed(b, which):
    rng = np.random.default_rng(17)
    full = rng.standard_normal((b.nbatch, b.layout.sol_stride))
    if which == "all":
        return full
    seed = np.zeros_like(full)
    for k in range(b.shape.N + 1):
        o, sz = b.layout.off[which][k], b.layout.size[which][k]
        seed[:, o:o + sz] = full[:, o:o + sz]
    return seed


def _check(b, e1, e2, adjoint, ok, s1, s2):
    """e2: a sensitivity record, or a function (q, fld) -> max |a1 - a2| / max |a2| over field fld of QP q."""
    L = b.layout
    lt1 = np.concatenate([L.gather(s1, "lam"), L.gather(s1, "t")], axis=1)
    lt2 = np.concatenate([L.gather(s2, "lam"), L.gather(s2, "t")], axis=1)
    agree = np.max(np.abs(lt1 - lt2) / np.maximum(np.abs(lt2), 1e-300), axis=1, initial=0.0)   # elementwise relative: Gamma = lam / t
    ntight = 0
    for q in np.nonzero(ok)[0]:
        tight = 1e-9 if agree[q] <= 1e-13 else 1e-2
        ntight += agree[q] <= 1e-13
        for fld in ("ux", "pi", "lam", "t"):
            if callable(e2):
                err = e2(q, fld)
            else:
                a1, a2 = L.gather(e1[q:q + 1], fld)[0], L.gather(e2[q:q + 1], fld)[0]
                err = np.max(np.abs(a1 - a2)) / max(np.max(np.abs(a2)), 1e-300) if a2.size else None
            if err is None:
                continue
            loose = fld == "lam" or (fld == "t" and adjoint)
            assert err <= (2e-2 if loose else tight), (q, fld, err, agree[q])
    return ntight


@pytest.mark.parametrize("name", SENS_CASES)
@pytest.mark.parametrize("adjoint", [False, True])
@pytest.mark.parametrize("which", ["ux", "lam", "all"])
def test_oracle_sens_matches_reference(built, name, adjoint, which):
    """The reference's solution is the golden one of tests/golden/<name>.npz (same solve); its sensitivities are compared on
    the stored sample of every field, relative to the field's max |.| as in the full comparison."""
    from oracle import oracle_binding as ob
    b = CASES[name]()
    seed = _seed(b, which)
    o = default_opts()
    s1, i1, e1 = ob.oracle_solve_sens(b, o, seed, adjoint=adjoint)
    z, key = reference_outputs("sens"), f"{name}/adj{int(adjoint)}/{which}"
    assert np.allclose(input_fingerprint(b.qp), z[name + "/inputs"], rtol=1e-12, atol=0), "generator drifted from the stored inputs"
    g = np.load(os.path.join(GOLD, name + ".npz"), allow_pickle=False)
    assert np.array_equal(i1["iter"], z[key + "/iter"])

    def err(q, fld):
        if key + f"/{fld}/idx" not in z:
            return None
        v2, eps = ref_decode(z, key + f"/{fld}/val")
        norm = z[key + f"/{fld}/norm"][q]
        a1 = b.layout.gather(e1[q:q + 1], fld)[0, z[key + f"/{fld}/idx"]]
        return np.max(np.abs(a1 / norm - v2[q])) + eps

    _check(b, e1, err, adjoint, g["status"] == 0, s1, g["sol"])


def test_sens_is_linear_in_the_seed(built):
    """Property: the sensitivity map is linear (same factorisation, two seeds and their combination)."""
    from oracle import oracle_binding as ob
    b = CASES["c2_chain_mass"]()
    o = default_opts()
    sa, sb = _seed(b, "ux"), _seed(b, "pi")
    _, _, ea = ob.oracle_solve_sens(b, o, sa)
    _, _, eb = ob.oracle_solve_sens(b, o, sb)
    _, _, ec = ob.oracle_solve_sens(b, o, 2.0 * sa - 3.0 * sb)
    ref = 2.0 * ea - 3.0 * eb
    assert np.max(np.abs(b.layout.gather(ec, "ux") - b.layout.gather(ref, "ux"))) <= 1e-9 * np.max(np.abs(ref))


@pytest.mark.gpu
@pytest.mark.parametrize("name", SENS_CASES)
@pytest.mark.parametrize("adjoint", [False, True])
@pytest.mark.parametrize("warps", [1, 4])
def test_cuda_sens_matches_oracle(built, name, adjoint, warps):
    from acados_b200.binding import CuipmSolver
    from oracle import oracle_binding as ob
    b = CASES[name]()
    seed = _seed(b, "all")
    o = default_opts()
    s = CuipmSolver(b.shape, b.nbatch)
    s.set_tuning("warps", warps)
    sol, info = s.solve(b.qp, o)
    e1 = s.sens(seed, o, adjoint=adjoint)
    s.close()
    osol, oinfo, e2 = ob.oracle_solve_sens(b, o, seed, adjoint=adjoint)
    assert np.array_equal(info["iter"], oinfo["iter"])
    _check(b, e1, e2, adjoint, oinfo["status"] == 0, sol, osol)


@pytest.mark.gpu
def test_cuda_sens_full_size_linearity(built):
    """BASELINE config 2 at batch 1024: sens(2a - 3b) = 2 sens(a) - 3 sens(b) on the device path, and the solution of the
    preceding solve is left untouched."""
    from acados_b200 import problems as P
    from acados_b200.binding import CuipmSolver
    b = P.chain_mass(1024, seed=4321)
    o = default_opts()
    s = CuipmSolver(b.shape, b.nbatch)
    sol, info = s.solve(b.qp, o)
    sa, sb = _seed(b, "ux"), _seed(b, "pi")
    ea, eb, ec = s.sens(sa, o), s.sens(sb, o), s.sens(2.0 * sa - 3.0 * sb, o)
    sol2, _ = s.solve(b.qp, o)
    s.close()
    ref = 2.0 * ea - 3.0 * eb
    ux = b.layout.gather(ref, "ux")
    # linear up to round-off times the conditioning of the linearised KKT systems (Gamma = lam / t up to 1e16)
    err = np.max(np.abs(b.layout.gather(ec, "ux") - ux), axis=1) / np.max(np.abs(ux), axis=1)
    assert np.median(err) <= 1e-12 and err.max() <= 1e-6, (np.median(err), err.max())
    assert np.array_equal(sol, sol2)
