"""GPU parity tests (run on the B200 box with -m gpu): the CUDA path, called through the C ABI, against
 (a) the plain-C oracle on the same seeded records, (b) the committed golden vectors produced by the reference,
 (c) stored outputs of the reference on a larger batch, and (d) size-independent properties at BASELINE.json's sizes.
Tolerance (north_star): |du|_inf <= 1e-10 on identical inputs, IPM iteration counts equal."""
import os

import numpy as np
import pytest

from acados_b200 import problems as P
from acados_b200.binding import CuipmSolver, default_opts
from test_oracle_vs_reference import CASES, GOLD, TOL_U

pytestmark = pytest.mark.gpu


def _solve(b, o, warps=None, **kw):
    s = CuipmSolver(b.shape, b.nbatch)
    if warps:
        s.set_tuning("warps", warps)
    out = s.solve(b.qp, o, **kw)
    s.close()
    return out


def _tol_default(name):
    """|du|_inf bar at the DEFAULT solver tolerances (1e-6/1e-8): the north_star's 1e-10 on the named workloads
    (mass-spring, chain-mass).  The synthetic random families stop ~1e-8 away from the exact solution with slack
    penalties up to 1e3, where summation-order round-off is amplified to a few 1e-10 (1.2e-10 observed between the
    CUDA path and the oracle on c5_sized); they are held to 1e-9 here and to 1e-10 in the tight-tolerance run below."""
    return TOL_U if name.startswith(("c1", "c2", "unconstrained")) else 1e-9


def _tol_default_at_size(name):
    """The same at the configurations' full batch sizes, where 64 instances are compared instead of a handful: the tail of the
    synthetic families reaches 1.1e-9 (c4, 8192) at the default tolerances; test_other_configs_at_size then drives the same
    instances to 1e-12 residuals and holds them to 1e-10."""
    return TOL_U if name.startswith(("c1", "c2")) else 5e-9


@pytest.mark.parametrize("name", list(CASES))
@pytest.mark.parametrize("warps", [1, 2, 4])
def test_cuda_matches_oracle(built, name, warps):
    from oracle import oracle_binding as ob
    b = CASES[name]()
    o = default_opts()
    sol, info, stat = _solve(b, o, warps, want_stat=True)
    osol, oinfo, ostat = ob.oracle_solve(b, o, want_stat=True)
    assert np.array_equal(info["iter"], oinfo["iter"]), (info["iter"], oinfo["iter"])
    assert np.array_equal(info["status"], oinfo["status"])
    # the switch to the LQ refactorisation is triggered by round-off (see test_oracle_vs_reference): +-1 iteration
    assert np.max(np.abs(info["lq_count"] - oinfo["lq_count"])) <= 1
    du = np.max(np.abs(b.layout.u_traj(sol) - b.layout.u_traj(osol)))
    assert du <= _tol_default(name), du
    assert np.max(np.abs(sol - osol)) <= 1e-6 * max(1.0, np.max(np.abs(osol)))
    for q in range(b.nbatch):
        it = info["iter"][q]
        same = info["lq_count"][q] == oinfo["lq_count"][q]
        assert np.allclose(stat[q, :it + 1, :13], ostat[q, :it + 1, :13], rtol=1e-4, atol=1e-6 if same else 1e-5)
        if same:
            assert np.array_equal(stat[q, :it + 1, 13], ostat[q, :it + 1, 13])
    assert np.allclose(info["obj"], oinfo["obj"], rtol=1e-9, atol=1e-9)


def _lq_compare(b, o, warps):
    from oracle import oracle_binding as ob
    sol, info, stat = _solve(b, o, warps, want_stat=True)
    osol, oinfo, ostat = ob.oracle_solve(b, o, want_stat=True)
    assert np.array_equal(info["iter"], oinfo["iter"]), (info["iter"], oinfo["iter"])
    assert np.array_equal(info["status"], oinfo["status"])
    assert np.max(np.abs(info["lq_count"] - oinfo["lq_count"])) <= (1 if o.lq_fact == 1 else 0), (info["lq_count"], oinfo["lq_count"])
    du = np.max(np.abs(b.layout.u_traj(sol) - b.layout.u_traj(osol)).reshape(b.nbatch, -1), axis=1)
    conv = oinfo["status"] == 0
    return du, conv, oinfo


@pytest.mark.parametrize("name", ["c1_mass_spring", "c2_chain_mass", "rand_general", "rand_soft", "rand_masked", "rand_x0_free", "c5_sized"])
@pytest.mark.parametrize("warps", [1, 4])
def test_cuda_lq_every_iteration(built, name, warps):
    """lq_fact = 2 (HPIPM ROBUST mode): every factorisation goes through the LQ sweep."""
    b = CASES[name]()
    du, conv, oinfo = _lq_compare(b, default_opts(lq_fact=2), warps)
    assert conv.all() and (oinfo["lq_count"] == oinfo["iter"]).all()
    assert du.max() <= _tol_default(name), du


@pytest.mark.parametrize("name", ["infeasible_box", "infeasible_general", "infeasible_soft"])
def test_cuda_lq_fallback(built, name):
    """Near-singular instances on which the Cholesky step fails the accuracy test and the solver refactorises with LQ
    (lq_fact = 1, the acados default): same trajectory as the oracle (pinned against the reference on these cases)."""
    from test_oracle_vs_reference import LQ_CASES
    b = LQ_CASES[name]()
    du, conv, oinfo = _lq_compare(b, default_opts(lq_fact=1), 1)
    assert (oinfo["lq_count"] > 0).sum() >= 8
    assert du[conv].max(initial=0.0) <= 1e-9 and du.max() <= 1e-7, du


@pytest.mark.parametrize("name", [n for n in CASES if n not in ("rand_infeasible", "c2_chain_hard")])
def test_cuda_matches_oracle_converged(built, name):
    """Both solvers driven to 1e-12 residuals: |du|_inf <= 1e-10 on every family (the stopping test may flip one
    iteration earlier/later at round-off-level tolerances; instances where it does are compared all the same)."""
    from oracle import oracle_binding as ob
    b = CASES[name]()
    o = default_opts(res_g_max=1e-12, res_b_max=1e-12, res_d_max=1e-12, res_m_max=1e-12)
    sol, info = _solve(b, o)
    osol, oinfo = ob.oracle_solve(b, o)
    assert np.max(np.abs(info["iter"] - oinfo["iter"])) <= 1
    ok = (info["status"] == 0) & (oinfo["status"] == 0)
    assert ok.all()
    assert np.max(np.abs(b.layout.u_traj(sol) - b.layout.u_traj(osol))) <= TOL_U


@pytest.mark.parametrize("name", sorted(f[:-4] for f in os.listdir(GOLD) if f.endswith(".npz") and not f.startswith("refjson_")))
def test_cuda_matches_golden_reference_vectors(built, name):
    g = np.load(os.path.join(GOLD, name + ".npz"), allow_pickle=False)
    b = CASES[str(g["case"])]()
    assert np.array_equal(np.asarray(b.qp[:, :64]), g["qp_head"])
    sol, info = _solve(b, default_opts())
    assert np.array_equal(info["iter"], g["iter"]) and np.array_equal(info["status"], g["status"])
    assert np.max(np.abs(b.layout.u_traj(sol) - g["u"])) <= _tol_default(name)


def test_cuda_matches_reference_when_present(built):
    """Against the reference's outputs for these QPs, stored by tests/golden/make_reference_outputs.py."""
    from test_oracle_vs_reference import stored_reference
    b = P.chain_mass(64, seed=77)
    o = default_opts()
    sol, info = _solve(b, o)
    r = stored_reference("gpu", "chain_mass64", b)
    ok = r["lq_count"] == 0
    assert ok.mean() > 0.9
    assert np.array_equal(info["iter"][ok], r["iter"][ok])
    u2, eps = r["u"]
    assert np.max(np.abs(b.layout.u_traj(sol) - u2)[ok]) + eps <= TOL_U


@pytest.mark.parametrize("ws", [2, 3])
def test_warm_start_parity(built, ws):
    from oracle import oracle_binding as ob
    b = P.chain_mass(8, N=12, seed=21)
    sol0, _ = ob.oracle_solve(b, default_opts())
    o = default_opts(warm_start=ws)
    sol, info = _solve(b, o, sol0=sol0)
    osol, oinfo = ob.oracle_solve(b, o, sol0=sol0)
    assert np.array_equal(info["status"], oinfo["status"])
    if ws == 2:
        assert np.array_equal(info["iter"], oinfo["iter"])
    else:
        # warm_start=3 restarts from the converged point with lam, t clipped at 1e-9: the first step drives lam + dlam to
        # zero up to round-off, and the ratio test (x_core_qp_ipm_aux.c:375-398) returns alpha = 1 or 1 - O(1e-7)
        # depending on the sign of that round-off.  alpha < 1 shortens the step (alpha*((1-alpha)*0.99+alpha*0.9999999))
        # and leaves 2e-7 of the initial residual (~1e2), i.e. above res_g_max: one more iteration.  The flip is a
        # discontinuity of the reference algorithm itself (the summation order of the Riccati sweeps decides it), so the
        # count may differ by one; status and solution are held to the same bars.
        assert np.max(np.abs(info["iter"] - oinfo["iter"])) <= 1, (info["iter"], oinfo["iter"])
    assert np.max(np.abs(b.layout.u_traj(sol) - b.layout.u_traj(osol))) <= (1e-9 if ws == 2 else 1e-7)


@pytest.mark.parametrize("name", ["c1_mass_spring", "c2_chain_mass", "rand_soft"])
def test_tau_min_parity(built, name):
    """acados' ``tau_min`` option (m != 0: relaxed complementarity target and the quadratic ratio test): CUDA path (generic kernel:
    the throughput kernel is bypassed for this option) against the oracle, which test_oracle_vs_reference pins to the reference."""
    from oracle import oracle_binding as ob
    b = CASES[name]()
    o = default_opts(m_relax=1e-3)
    sol, info = _solve(b, o)
    osol, oinfo = ob.oracle_solve(b, o)
    assert np.array_equal(info["status"], oinfo["status"]) and np.array_equal(info["iter"], oinfo["iter"]), (info["iter"], oinfo["iter"])
    conv = oinfo["status"] == 0
    assert np.max(np.abs(b.layout.u_traj(sol) - b.layout.u_traj(osol))[conv], initial=0.0) <= _tol_default(name)


def test_tight_tolerance_parity(built):
    """Both solvers driven to 1e-12 residuals: solutions agree far below the 1e-10 bar (iteration count may flip by one)."""
    from oracle import oracle_binding as ob
    b = P.chain_mass(16, seed=9)
    o = default_opts(res_g_max=1e-12, res_b_max=1e-12, res_d_max=1e-12, res_m_max=1e-12)
    sol, info = _solve(b, o)
    osol, oinfo = ob.oracle_solve(b, o)
    assert np.max(np.abs(info["iter"] - oinfo["iter"])) <= 1
    same = info["iter"] == oinfo["iter"]
    assert np.max(np.abs(b.layout.u_traj(sol) - b.layout.u_traj(osol))[same]) <= 1e-11


def test_full_size_properties_c2(built):
    """BASELINE config 2 at full size (batch 4096): every instance converges, independently recomputed KKT
    residuals are within the solver tolerances, results do not depend on the position in the batch, and a second
    run is bit-identical."""
    from oracle import oracle_binding as ob
    b = P.chain_mass(4096, seed=1234)
    o = default_opts()
    s = CuipmSolver(b.shape, b.nbatch)
    sol, info = s.solve(b.qp, o)
    assert (info["status"] == 0).all()
    assert info["iter"].max() <= 30 and info["iter"].min() >= 3
    r = ob.oracle_residuals(b, sol)
    assert (r["res_max"][:, 0] <= o.res_g_max).all(), r["res_max"][:, 0].max()
    assert (r["res_max"][:, 1] <= o.res_b_max).all(), r["res_max"][:, 1].max()
    assert (r["res_max"][:, 2] <= o.res_d_max).all(), r["res_max"][:, 2].max()
    assert (r["res_max"][:, 3] <= o.res_m_max + 1e-9).all(), r["res_max"][:, 3].max()
    assert np.allclose(r["obj"], info["obj"], rtol=1e-10, atol=1e-10)
    # spot-check a slice against the oracle
    idx = np.arange(0, 4096, 128)
    sub = P.Batch(b.shape, b.layout, np.ascontiguousarray(b.qp[idx]))
    osol, oinfo = ob.oracle_solve(sub, o)
    assert np.array_equal(info["iter"][idx], oinfo["iter"])
    # At the DEFAULT tolerances (1e-6/1e-8) both solvers stop ~1e-8 from the exact solution and summation-order round-off
    # decides the last digits: 98.7 % of the 4096 instances are within the north_star's 1e-10, the largest difference seen
    # over the whole batch is 2.1e-9 (bench.py's parity record) -- a property of where the iteration stops, not of the
    # arithmetic.  The 1e-10 bar itself is asserted on ALL 4096 instances at tight tolerances in
    # test_tight_tolerance_parity_full_headline_batch; here the slice is held to "bulk within 1e-10, nothing beyond 5e-9".
    d = np.max(np.abs(b.layout.u_traj(sol[idx]) - b.layout.u_traj(osol)), axis=1)
    assert (d <= TOL_U).mean() >= 0.9 and d.max() <= 5e-9, (d.max(), (d <= TOL_U).mean())
    # batch-position independence + determinism
    perm = np.random.default_rng(0).permutation(4096)
    sol_p, info_p = s.solve(np.ascontiguousarray(b.qp[perm]), o)
    assert np.array_equal(info_p["iter"], info["iter"][perm])
    assert np.array_equal(sol_p, sol[perm]), f"position dependence: max diff {np.max(np.abs(sol_p - sol[perm]))}"
    sol2, _ = s.solve(b.qp, o)
    assert np.array_equal(sol2, sol)
    s.close()


def test_tight_tolerance_parity_full_headline_batch(built):
    """BASELINE.md section 4: all tolerances 1e-12 on the WHOLE headline batch (chain-mass, 4096 instances), CUDA path against
    the reference (oracle/_ref when it travelled, else the oracle port): |du|_inf <= 1e-10 on every instance -- the north_star's
    bar -- and iteration counts within one (the last iteration is decided by residuals at round-off level)."""
    from oracle import oracle_binding as ob
    b = P.chain_mass(4096, seed=1234)
    o = default_opts(res_g_max=1e-12, res_b_max=1e-12, res_d_max=1e-12, res_m_max=1e-12)
    sol, info = _solve(b, o)
    from acados_b200.binding import host_threads
    nt = host_threads()
    if ob.have_ref():
        rsol, rinfo, _ = ob.ref_solve(b, o, nthreads=nt)
    else:
        rsol, rinfo = ob.oracle_solve(b, o, nthreads=nt)
    assert np.array_equal(info["status"], rinfo["status"]) and (info["status"] == 0).all()
    assert np.max(np.abs(info["iter"] - rinfo["iter"])) <= 1
    du = np.max(np.abs(b.layout.u_traj(sol) - b.layout.u_traj(rsol)), axis=1)
    assert du.max() <= 1e-10, (du.max(), int((du > 1e-10).sum()))


@pytest.mark.parametrize("name,nb", [("c3", 16384), ("c4", 8192), ("c5", 1024)])
def test_other_configs_at_size(built, name, nb):
    from oracle import oracle_binding as ob
    b = P.named_config(name, nb)
    o = default_opts()
    sol, info = _solve(b, o)
    assert (info["status"] == 0).mean() > 0.98
    from acados_b200.binding import host_threads
    nt = host_threads()
    idx = np.arange(0, nb, max(1, nb // 64))
    sub = P.Batch(b.shape, b.layout, np.ascontiguousarray(b.qp[idx]))
    osol, oinfo = ob.oracle_solve(sub, o, nthreads=min(16, nt))
    assert np.array_equal(info["iter"][idx], oinfo["iter"])
    assert np.max(np.abs(b.layout.u_traj(sol[idx]) - b.layout.u_traj(osol))) <= _tol_default_at_size(name)
    # the north_star's bar on the same instances with both solvers driven to 1e-12 residuals
    ot = default_opts(res_g_max=1e-12, res_b_max=1e-12, res_d_max=1e-12, res_m_max=1e-12)
    tsol, tinfo = _solve(sub, ot)
    tosol, toinfo = ob.oracle_solve(sub, ot, nthreads=min(16, nt))
    conv = (tinfo["status"] == 0) & (toinfo["status"] == 0)
    # (at 1e-12 the last iterations are decided by residuals at round-off level: counts within two on the synthetic families)
    assert conv.mean() > 0.9 and np.max(np.abs(tinfo["iter"] - toinfo["iter"])[conv]) <= 2
    assert np.max(np.abs(b.layout.u_traj(tsol) - b.layout.u_traj(tosol))[conv]) <= TOL_U


@pytest.mark.parametrize("case", ["c2", "c4", "soft_masked"])
def test_iteration_sliced_scheduling_gpu(built, case):
    """The throughput kernel's two schedules -- a QP bound to its warp for the whole solve (tuning rr=0), or for one iteration at a
    time with the unfinished QPs circulating through a ring (rr=2: forced; the default switches it on when the batch exceeds the
    resident QPs) -- run the same arithmetic on the same records: solutions and summaries are bit-identical, whatever the order in
    which QPs meet in a warp.  The last case has QPs that are handed back to the generic kernel."""
    if case == "c2":
        b = P.chain_mass(4096, seed=1234)
    elif case == "c4":
        b = P.named_config("c4", 3000)
    else:
        b = P.random_qp(P.random_shape(12, 8, 3, nbx=4, ns=2), 3000, seed=5, mask_frac=0.3)
    o = default_opts()
    s = CuipmSolver(b.shape, b.nbatch)
    out = {}
    for rr in (2, 0):
        s.set_tuning("rr", rr)
        out[rr] = s.solve(b.qp, o)
        out[rr] = (out[rr][0], out[rr][1], s.last_launch_count, s.last_handed_back)
    s.close()
    assert out[2][2] > out[0][2]                            # one more launch per chunk: rr_first + rr_loop instead of the single kernel
    assert np.array_equal(out[2][0], out[0][0])
    for f in ("status", "iter", "mu", "obj", "dual_gap", "res_max", "lq_count"):
        assert np.array_equal(out[2][1][f], out[0][1][f]), f
    assert out[2][3] == out[0][3]
    if case == "soft_masked":
        assert out[0][3] > 0


def test_edge_cases(built):
    from oracle import oracle_binding as ob
    o = default_opts()
    # empty batch, batch of one, horizon of one
    s = CuipmSolver(P.mass_spring(1).shape, 4)
    sol, info = s.solve(np.zeros((0, s.layout.qp_stride)), o)
    assert sol.shape[0] == 0
    with pytest.raises(RuntimeError):
        s.solve(P.mass_spring(5).qp, o)      # larger than max_batch
    s.close()
    b = P.random_qp(P.random_shape(1, 3, 2, nbx=2), 3, seed=3, umax=0.5, xmax=3.0)
    sol, info = _solve(b, o)
    osol, oinfo = ob.oracle_solve(b, o)
    assert np.array_equal(info["iter"], oinfo["iter"]) and np.max(np.abs(sol - osol)) < 1e-9
    # iteration limit and unsupported options
    b = P.chain_mass(4, N=8, seed=2)
    sol, info = _solve(b, default_opts(iter_max=2))
    assert (info["status"] == 1).all() and (info["iter"] == 2).all()
    with pytest.raises(RuntimeError, match="not supported"):
        _solve(b, default_opts("SPEED"))


def test_riccati_getters(built):
    """P, p, K, k, Lr of the last factorisation (reference getters ocp_qp_hpipm.c:417-478) on an unconstrained LQR:
    u_0 = K_0 x_0 + k_0 must reproduce the solution and P must be symmetric positive definite."""
    b = P.random_qp(P.random_shape(6, 4, 2, nbu=0, x0_eliminated=False), 2, seed=4)
    s = CuipmSolver(b.shape, b.nbatch)
    sol, info = s.solve(b.qp, default_opts())
    for q in range(b.nbatch):
        for k in range(0, 6):
            nx, nu = b.shape.nx[k], b.shape.nu[k]
            K = s.get_ric(q, "K", k, (nu, nx)); kk = s.get_ric(q, "k", k, (nu, 1)).ravel()
            Pm = s.get_ric(q, "P", k, (nx, nx))
            ux = b.layout.view(sol, "ux", k)[q]
            assert np.allclose(K @ ux[nu:nu + nx] + kk, ux[:nu], atol=1e-9)
            assert np.allclose(Pm, Pm.T) and (np.linalg.eigvalsh(Pm) > 0).all()
            Lr = s.get_ric(q, "Lr", k, (nu, nu))
            assert np.allclose(np.triu(Lr, 1), 0) and (np.diag(Lr) > 0).all()
    s.close()


def test_async_host_entry_matches_blocking(built):
    """cuipm_solve_host_async / cuipm_wait on two solver objects used alternately (the double buffering of bench.py's
    end-to-end leg): bit-identical to the blocking entry, whatever is in flight on the other object."""
    import torch
    b = P.chain_mass(1024, seed=99)
    o = default_opts()
    ref_sol, ref_info = _solve(b, o)
    solvers = [CuipmSolver(b.shape, b.nbatch) for _ in range(2)]
    h_qp = torch.from_numpy(b.qp).pin_memory()
    outs = [(torch.zeros((b.nbatch, b.layout.sol_stride), dtype=torch.float64).pin_memory(),
             torch.zeros(b.nbatch * ref_info.dtype.itemsize, dtype=torch.uint8).pin_memory()) for _ in range(2)]
    for i in range(5):
        s, (hs, hi) = solvers[i % 2], outs[i % 2]
        s.wait()
        s.solve_host_async(b.nbatch, h_qp.data_ptr(), hs.data_ptr(), hi.data_ptr(), o)
    for s in solvers:
        s.wait()
    for hs, hi in outs:
        assert np.array_equal(hs.numpy(), ref_sol)
        assert np.array_equal(np.frombuffer(hi.numpy().tobytes(), dtype=ref_info.dtype)["iter"], ref_info["iter"])
    for s in solvers:
        s.close()
