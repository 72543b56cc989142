"""The CPU oracle (oracle_kin.c) on the DH-like chains of oracle.chains.dh_like_chain, against an extended-precision
restatement.

tests/test_gpu_fkj_joint_counts.py checks the kernels against the oracle on these chains for n = 1..10, shapes no golden
fixture covers, so the oracle itself is pinned here first.  The restatement works in np.longdouble (64-bit mantissa on
x86-64) straight from the chain description:
  T  = base . A_0 Rz(q_0) A_1 Rz(q_1) ... Rz(q_{n-1}) A_n . tool, the constants and Rz(q_j) as 4x4 products;
  J0 column j = [z_j x (p_e - p_j); z_j], z_j / p_j the axis and origin of joint j (no base, tool included);
  Je = blkdiag(R^T, R^T) . J0, R the rotation of the pose without the base.
"""
import numpy as np
import pytest

from oracle import chains as ch
from oracle import oracle as orc

LD = np.longdouble


def rz(q):
    """Rz(q_k) for a vector of angles: (N, 4, 4) in long double."""
    c, s = np.cos(q), np.sin(q)
    R = np.zeros((q.shape[0], 4, 4), dtype=LD)
    R[:, 0, 0], R[:, 0, 1], R[:, 1, 0], R[:, 1, 1] = c, -s, s, c
    R[:, 2, 2] = R[:, 3, 3] = 1
    return R


def reference(desc, Q, base=None, tool=None):
    """(T, J0, Je) of every row of Q in long double."""
    N = Q.shape[0]
    q = Q.astype(LD)
    M = np.broadcast_to(np.eye(4, dtype=LD), (N, 4, 4)).copy()
    z, p = [], []
    for isjoint, axis, flip, jindex, A in zip(desc["isjoint"], desc["axis"], desc["flip"], desc["jindex"], desc["T"]):
        if not isjoint:
            M = M @ A.astype(LD)
            continue
        assert axis == ch.RZ and not flip, "the restatement covers DH-like chains only"
        z.append(M[:, :3, 2].copy())
        p.append(M[:, :3, 3].copy())
        M = M @ rz(q[:, jindex])
    if tool is not None:
        M = M @ np.asarray(tool).astype(LD)
    pe = M[:, :3, 3]
    J0 = np.zeros((N, 6, len(z)), dtype=LD)
    for j, (zj, pj) in enumerate(zip(z, p)):
        J0[:, :3, j] = np.cross(zj, pe - pj)
        J0[:, 3:, j] = zj
    Rt = M[:, :3, :3].transpose(0, 2, 1)
    Je = np.concatenate([Rt @ J0[:, :3], Rt @ J0[:, 3:]], axis=1)
    T = M if base is None else np.asarray(base).astype(LD) @ M
    return T, J0, Je


def inputs(rng, N, n):
    """Mostly U(-pi, pi); a tenth of the rows with angles in [8, 100) and a tenth with one joint beyond 1.1e5."""
    Q = rng.uniform(-np.pi, np.pi, (N, n))
    mid = rng.choice(N, N // 10, replace=False)
    Q[mid] = rng.uniform(8, 100, (mid.size, n)) * rng.choice([-1, 1], (mid.size, n))
    huge = rng.choice(np.setdiff1d(np.arange(N), mid), N // 10, replace=False)
    Q[huge, rng.integers(0, n, huge.size)] = rng.uniform(1.1e5, 1e6, huge.size) * rng.choice([-1, 1], huge.size)
    return Q


@pytest.mark.parametrize("tail", [False, True])
@pytest.mark.parametrize("n", range(1, 11))
def test_oracle_matches_long_double_on_dh_like_chains(n, tail):
    rng = np.random.default_rng(1000 * n + tail)
    desc = ch.dh_like_chain(rng, n, tail=tail)
    C = orc.Chain(desc)
    base, tool = ch.random_se3(rng), ch.random_se3(rng)
    Q = inputs(rng, 400, n)
    for b, t in ((None, None), (base, tool)):
        tol = dict(rtol=1e-13, atol=1e-13 * max(1.0, ch.chain_reach(desc, b, t)))
        T, J0, Je = (x.astype(np.float64) for x in reference(desc, Q, b, t))
        np.testing.assert_allclose(C.fkine(Q, b, t), T, **tol)
        np.testing.assert_allclose(C.jacob0(Q, t), J0, **tol)
        np.testing.assert_allclose(C.jacobe(Q, t), Je, **tol)


def test_generator_shapes():
    """The generator draws what the GPU tests rely on: n unflipped Rz joints, Rx-form inter-joint constants with
    alpha = 0 and +-pi/2 among them, and a constant after the last joint exactly when a tail is asked for."""
    alphas = set()
    for n in range(1, 11):
        for tail in (False, True):
            d = ch.dh_like_chain(np.random.default_rng(n), n, tail=tail)
            isj = d["isjoint"].astype(bool)
            assert d["n"] == n and (d["axis"][isj] == ch.RZ).all() and not d["flip"].any()
            assert bool(isj[-1]) != tail and not isj[0]
            for k in np.flatnonzero(isj)[:-1]:
                A = d["T"][k + 1]
                assert A[0, 0] == 1 and A[0, 1] == A[0, 2] == A[1, 0] == A[2, 0] == 0  # Rx form, as b2k_classify34 tests it
                alphas.add(round(float(np.arctan2(A[2, 1], A[1, 1])), 12))
    assert {0.0, round(np.pi / 2, 12), round(-np.pi / 2, 12)} <= alphas
