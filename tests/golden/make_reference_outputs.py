"""Generates tests/golden/reference/*.npz.xz: what the unmodified reference (oracle/_ref, built from the reference sources by
oracle/Makefile) returns for the inputs of the tests that compare against it, so that those comparisons run on any machine.
  python tests/golden/make_reference_outputs.py

Storage.  Integer arrays, and the solutions the warm-start tests restart from, are stored as they are.  A float array x is stored as x_hat = base + h * q with integer q, where base is
zero, another stored array or an array of the golden files next to this script, and h is a resolution chosen three orders of
magnitude below the tolerance the test applies to x; eps = max|x_hat - x| is stored with it.  A test that asserts
|a - x| <= tol checks |a - x_hat| + eps <= tol instead, which implies it (see ref_decode in test_oracle_vs_reference.py).
The per-iteration statistics span many magnitudes and are held to a relative tolerance: they are stored in float32 with
their relative rounding bound.
Outputs of the same solve under another option are stored against the first one as base, so near-identical arrays cost
almost nothing.  The sensitivity records are sampled: one entry per stage and SENS_SAMPLES more per field and QP, divided by
the field's max |.|, which is stored exactly.
"""
import io
import lzma
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from acados_b200 import problems as P  # noqa: E402
from acados_b200.binding import default_opts  # noqa: E402
from oracle import oracle_binding as ob  # noqa: E402
from test_oracle_vs_reference import CASES, GOLD, LQ_CASES, REF_OUT, TOL_U, input_fingerprint, ref_decode  # noqa: E402

SENS_SAMPLES = 8


def _int(x):
    x = np.asarray(x)
    for t in (np.int8, np.int16, np.int32, np.int64):
        if np.all(np.abs(x) <= np.iinfo(t).max):
            assert np.array_equal(x, x.astype(t))
            return x.astype(t)
    raise ValueError("out of range")


class Store(dict):
    def exact(self, key, x):
        self[key] = np.asarray(x)

    def approx(self, key, x, h, base=None):
        x = np.asarray(x, dtype=np.float64)
        b = 0.0 if base is None else ref_decode(self, base)[0]
        q = np.round((x - b) / h)
        assert np.all(np.abs(q) < 2.0 ** 62), key
        self[key + ".q"], self[key + ".h"] = _int(q), np.float64(h)
        if base is not None:
            self[key + ".base"] = np.array(base)
        self[key + ".eps"] = np.float64(0.0)
        self[key + ".eps"] = np.float64(np.max(np.abs(ref_decode(self, key)[0] - x), initial=0.0))

    def relative(self, key, x):
        """float32 with the relative bound r = max |x_hat - x| / |x| (for values of many magnitudes held to a relative tolerance)."""
        x = np.asarray(x, dtype=np.float64)
        self[key + ".f32"] = x.astype(np.float32)
        err = np.abs(self[key + ".f32"].astype(np.float64) - x)
        self[key + ".rel"] = np.float64(np.max(np.where(err > 0, err / np.maximum(np.abs(x), 1e-300), 0.0), initial=0.0))

    def save(self, group):
        """One uncompressed .npz compressed as a whole with xz: most arrays are small, and their headers compress with them."""
        buf = io.BytesIO()
        np.savez(buf, **self)
        os.makedirs(REF_OUT, exist_ok=True)
        path = os.path.join(REF_OUT, group + ".npz.xz")
        with open(path, "wb") as f:
            f.write(lzma.compress(buf.getvalue(), preset=9 | lzma.PRESET_EXTREME))
        print(f"{path}: {len(self)} arrays, {os.path.getsize(path)} bytes")


def solve_record(st, key, b, o, base=None, stats=True, sol0=None):
    """iter / status / lq_count, the input trajectory (1e-10 bar), the solution record (1e-6 relative bar) and the per-iteration
    statistics (rtol 1e-4) of one reference solve."""
    if stats:
        s, i, stat, _ = ob.ref_solve(b, o, want_stat=True, nthreads=1, sol0=sol0)
    else:
        s, i, _ = ob.ref_solve(b, o, nthreads=1, sol0=sol0)
    st.exact(key + "/iter", _int(i["iter"]))
    st.exact(key + "/status", _int(i["status"]))
    st.exact(key + "/lq_count", _int(i["lq_count"]))
    st.approx(key + "/u", b.layout.u_traj(s), 1e-3 * TOL_U, base and base + "/u")
    if stats:
        st.approx(key + "/sol", s, 1e-9 * max(1.0, np.max(np.abs(s))), base and base + "/sol")
        rows = np.concatenate([stat[q, :i["iter"][q] + 1] for q in range(b.nbatch)])
        st.relative(key + "/stat13", rows[:, :13])
        st.exact(key + "/lqflag", _int(rows[:, 13]))
    return s, i


def oracle_group():
    st = Store()
    for name, make in CASES.items():
        b = make()
        st.exact(name + "/inputs", input_fingerprint(b.qp))
        solve_record(st, name + "/lq1", b, default_opts(lq_fact=1), base=f"golden:{name}")
        for lq in (0, 2):
            solve_record(st, f"{name}/lq{lq}", b, default_opts(lq_fact=lq), base=name + "/lq1")
    for name in ("c1_mass_spring", "c2_chain_mass", "rand_soft", "rand_masked"):
        b = CASES[name]()
        for tau in (1e-4, 1e-2):
            solve_record(st, f"{name}/tau{tau:g}", b, default_opts(m_relax=tau), base=f"golden:{name}", stats=False)
    for name, make in LQ_CASES.items():
        b = make()
        st.exact(name + "/inputs", input_fingerprint(b.qp))
        solve_record(st, name, b, default_opts(lq_fact=1))
    b = P.chain_mass(4, N=12, seed=21)
    st.exact("warm/inputs", input_fingerprint(b.qp))
    for tight in (False, True):
        kw = dict(res_g_max=1e-12, res_b_max=1e-12, res_d_max=1e-12, res_m_max=1e-12) if tight else {}
        key = f"warm/tight{int(tight)}"
        s2, _ = solve_record(st, key, b, default_opts(**kw), stats=False)
        # the warm starts begin at the cold solution itself: stored exactly, the test hands it to the oracle unchanged
        st.exact(key + "/sol0", s2)
        for ws in (2, 3):
            solve_record(st, f"{key}/ws{ws}", b, default_opts(warm_start=ws, **kw), base=key, stats=False, sol0=s2)
    st.save("oracle")


def condensing_group():
    from test_condensing import _reference
    from test_ocp_qp_mirror import random_ocp_qp
    st = Store()
    for soft, general in ((False, False), (True, False), (True, True)):
        rng = np.random.default_rng(5)
        qps = [random_ocp_qp(rng, N=12, soft=soft, general=general) for _ in range(4)]
        base = None
        for cond_N in (12, 6, 5, 3, 1):
            full, rsol, rinfo = _reference(qps, cond_N, default_opts())
            key = f"soft{int(soft)}_general{int(general)}/N{cond_N}"
            st.exact(key + "/inputs", input_fingerprint(full.qp))
            st.exact(key + "/iter", _int(rinfo["iter"]))
            st.exact(key + "/status", _int(rinfo["status"]))
            st.approx(key + "/sol", rsol, 1e-3 * TOL_U, base)
            base = base or key + "/sol"
    st.save("condensing")


def _sens_sample(L, fld):
    """Columns of the gathered field: one seeded entry in every stage where it is not empty, and SENS_SAMPLES more anywhere."""
    rng = np.random.default_rng(23)
    sizes = [L.size[fld][k] for k in range(L.shape.N + 1)]
    starts = np.cumsum([0] + sizes[:-1])
    per_stage = [o + rng.integers(n) for o, n in zip(starts, sizes) if n > 0]
    extra = rng.choice(sum(sizes), min(SENS_SAMPLES, sum(sizes)), replace=False)
    return np.unique(np.concatenate([per_stage, extra]).astype(np.int64))


def sens_group():
    from test_sensitivities import SENS_CASES, _seed
    st = Store()
    for name in SENS_CASES:
        b = CASES[name]()
        L = b.layout
        st.exact(name + "/inputs", input_fingerprint(b.qp))
        for adjoint in (False, True):
            for which in ("ux", "lam", "all"):
                s2, i2, e2 = ob.ref_solve_sens(b, default_opts(), _seed(b, which), adjoint=adjoint)
                # the test takes the solution these sensitivities were evaluated at from the golden file of the case
                assert np.array_equal(s2, np.load(os.path.join(GOLD, name + ".npz"))["sol"])
                key = f"{name}/adj{int(adjoint)}/{which}"
                st.exact(key + "/iter", _int(i2["iter"]))
                for fld in ("ux", "pi", "lam", "t"):
                    a2 = L.gather(e2, fld)
                    if a2.shape[1] == 0:
                        continue
                    idx = _sens_sample(L, fld)
                    norm = np.maximum(np.max(np.abs(a2), axis=1), 1e-300)
                    st.exact(f"{key}/{fld}/idx", _int(idx))
                    st.exact(f"{key}/{fld}/norm", norm)
                    loose = fld == "lam" or (fld == "t" and adjoint)       # held to 2e-2 by the test, the others to 1e-9
                    st.approx(f"{key}/{fld}/val", a2[:, idx] / norm[:, None], 1e-3 * (2e-2 if loose else 1e-9))
    st.save("sens")


def gpu_group():
    st = Store()
    b = P.chain_mass(64, seed=77)
    st.exact("chain_mass64/inputs", input_fingerprint(b.qp))
    solve_record(st, "chain_mass64", b, default_opts(), stats=False)
    st.save("gpu")


if __name__ == "__main__":
    assert ob.have_ref(), "build oracle/_ref first: make -C oracle"
    oracle_group()
    condensing_group()
    sens_group()
    gpu_group()
