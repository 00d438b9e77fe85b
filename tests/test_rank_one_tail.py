"""The task tail of the fused kernel for a one-dimensional null space (a six-dof MotionForceTask over a 7-joint robot,
with a full JointTask below it: null vector of J instead of a Householder QR) against the QR prototype fast_cycle,
on the CPU."""
import numpy as np
import pytest

from oracle.robots import make_chain
from oracle.sai_model import SaiModel
from tests.algebra_proto import BIE, FULL, IMP, fast_cycle
from tests.osc_testlib import TASK_POINTS, rng_for

DECS = [FULL, BIE, IMP]


def rank_one_cycle(M, J, fstar, F, acc, t, dec_mft, bie_mft, dec_jt, bie_jt, use_prev=True):
    """Restatement of the fused kernel's task tail for a six-dof MotionForceTask (J: 6 x 7, full range) with a full
    JointTask in its one-dimensional null space: no QR, only the null vector n of J.
      G = J J^T = C C^T; n = column k* of I - J^T G^-1 J, k* = argmax of its diagonal 1 - |C^-1 J_k|^2;
      tau_task = M_b v - M_b n (n . M_b v) / (n . M_b n) + J^T F,  v = J^T G^-1 f  (impedance: J^T f + J^T F);
      tau_jt = M n [(n . acc - m . tau_task) / (n . n) + (n . t) / ((n . n) h)],  m = M^-1 n,
    h = 1 (full), 1 - delta n_e^2 / (s (1 + delta mu)) with one clamped entry e (s = n . M n, mu = |L^-1 e|^2);
    impedance: (n . t) / s.  Returns (tau, ok) with ok = not UNHANDLED: (n . n)(M n . M n) < 1e6 s^2."""
    n = M.shape[0]
    assert J.shape == (n - 1, n)
    L = np.linalg.cholesky(M)
    C = np.linalg.cholesky(J @ J.T)
    U = np.linalg.solve(C, J)                                   # C^-1 J_k, column by column
    k = int(np.argmax(1.0 - np.einsum("ak,ak->k", U, U)))
    nv = -J.T @ np.linalg.solve(C.T, U[:, k]); nv[k] += 1.0
    y = fstar if dec_mft == IMP else np.linalg.solve(C.T, np.linalg.solve(C, fstar))
    v = J.T @ y
    d = np.maximum(bie_mft - np.diag(M), 0.0) if dec_mft == BIE else np.zeros(n)
    Mbv = M @ v + d * v
    Mbn = M @ nv + d * nv
    tau = (v if dec_mft == IMP else Mbv - Mbn * (nv @ Mbv) / (nv @ Mbn)) + J.T @ F
    Mn = M @ nv
    s, nn = nv @ Mn, nv @ nv
    m = np.linalg.solve(L.T, np.linalg.solve(L, nv))
    zp = 1.0 / nn
    if dec_jt == IMP:
        zp = 1.0 / s
    elif dec_jt == BIE:
        dj = np.maximum(bie_jt - np.diag(M), 0.0)
        if np.count_nonzero(dj) == 1:
            e = int(np.argmax(dj)); delta = dj[e]
            g = np.linalg.solve(L, np.eye(n)[e]); mu = g @ g
            zp = zp / (1.0 - delta * nv[e] ** 2 / (s * (1.0 + delta * mu)))
        else:
            assert np.count_nonzero(dj) == 0, "two or more clamped entries leave for the general path"
    z = (nv @ acc - (m @ tau if use_prev else 0.0)) / nn + (nv @ t) * zp
    ok = nn * (Mn @ Mn) < 1e6 * s * s
    return tau + Mn * z, ok


def reference(M, J, fstar, F, acc, t, dm, bm, dj, bj, use_prev):
    mft = dict(kind="mft", B=np.eye(6), J0=J, fstar=fstar, F=F, dec=dm, bie=bm)
    jt = dict(kind="jt", S=np.eye(M.shape[0]), acc=acc, t=t, dec=dj, bie=bj)
    full, ok = fast_cycle(M, [mft, jt], None, None)
    if use_prev:
        return full
    # without the previous-torque term: drop the joint task's response to the task torque (-K z_dist in fast_cycle)
    jt0 = dict(jt, acc=np.zeros_like(acc), t=np.zeros_like(t))
    return full - fast_cycle(M, [mft, jt0], None, None)[0] + fast_cycle(M, [mft], None, None)[0]


def one_clamp_threshold(M):
    return np.sort(np.diag(M))[1] * 0.999   # exactly one diagonal entry below it


@pytest.mark.parametrize("use_prev", [True, False])
@pytest.mark.parametrize("dj", DECS)
@pytest.mark.parametrize("dm", DECS)
def test_rank_one_tail_equals_qr_route_on_random_cases(dm, dj, use_prev):
    g = rng_for(3 * dm + dj + 9 * use_prev, stream=31)
    n = 7
    for trial in range(100):
        A = g.normal(size=(n, n)); M = A @ A.T / n + np.diag(g.uniform(0.005, 0.5, n))
        J = g.normal(size=(6, n))
        fstar = g.normal(size=6); F = g.normal(size=6) * (trial % 2)
        acc = g.normal(size=n); t = g.normal(size=n)
        bm = one_clamp_threshold(M) if dm == BIE else 0.0
        bj = one_clamp_threshold(M) if dj == BIE else 0.0
        ref = reference(M, J, fstar, F, acc, t, dm, bm, dj, bj, use_prev)
        tau, _ = rank_one_cycle(M, J, fstar, F, acc, t, dm, bm, dj, bj, use_prev)
        assert np.abs(tau - ref).max() <= 1e-10 * np.abs(ref).max()


def panda_band_edge_states(count, lo=0.06, hi=0.07):
    """Panda states whose task Jacobian has s_min / s_max just above the 0.06 band of the fast path."""
    ch = make_chain("panda"); r = SaiModel(ch); n = ch.n
    link, pt = TASK_POINTS["panda"]
    g = rng_for(0, stream=32)
    found = []
    for trial in range(20000):
        q = ch.q_lower + (0.05 + 0.9 * g.random(n)) * (ch.q_upper - ch.q_lower)
        r.setQ(q); r.setDq(np.zeros(n)); r.updateModel()
        J = r.JWorldFrame(link, pt)
        s = np.linalg.svd(J, compute_uv=False)
        if lo < s[-1] / s[0] < hi:
            found.append((r.M().copy(), J.copy()))
            if len(found) == count:
                break
    assert len(found) == count
    return found


@pytest.mark.parametrize("use_prev", [True, False])
@pytest.mark.parametrize("dec", DECS)
def test_rank_one_tail_equals_qr_route_on_panda_band_edge(dec, use_prev):
    g = rng_for(dec + 3 * use_prev, stream=33)
    for M, J in panda_band_edge_states(12):
        n = M.shape[0]
        fstar = g.normal(size=6) * 10; F = g.normal(size=6)
        acc = g.normal(size=n); t = g.normal(size=n) * 10
        b = 0.1 if dec == BIE else 0.0   # the default threshold: one clamped entry on the Panda
        ref = reference(M, J, fstar, F, acc, t, dec, b, dec, b, use_prev)
        tau, ok = rank_one_cycle(M, J, fstar, F, acc, t, dec, b, dec, b, use_prev)
        assert ok
        assert np.abs(tau - ref).max() <= 1e-10 * np.abs(ref).max()
