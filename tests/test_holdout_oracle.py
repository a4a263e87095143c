"""The masked-step oracle (tests/holdout_oracle) and holdout.split_pairs on the CPU.

Where no clamp binds, the masked step is the BigCLAM objective with the held-out pairs left out of both terms:

    l_mask(F) = sum_{(u,v) in E_train} log(1 - exp(-Fu.Fv)) - sum_{u<v, (u,v) not in E_train u HO} Fu.Fv

evaluated here directly over all pairs (as tests/test_oracle_formula.py does for the unmasked objective): the masked LLH is
2 l_mask(F), the PRE gradient is grad_u l_mask(F), and the held-out LLH is the direct sum over the held-out pairs."""
import numpy as np
import pytest

from conftest import random_graph
from holdout_oracle import masked as M


def _split(rp, col, frac, seed):
    from bigclam_apachespark_b200.holdout import split_pairs
    return split_pairs(rp, col, frac, seed)


def _dense(n, rp, col):
    A = np.zeros((n, n), dtype=bool)
    for u in range(n):
        A[u, col[rp[u]:rp[u + 1]]] = True
    return A


@pytest.mark.parametrize("n,deg,k,seed", [(40, 6, 4, 1), (30, 8, 5, 2), (16, 10, 3, 3)])
def test_masked_oracle_is_the_masked_objective_where_no_clamp_binds(n, deg, k, seed):
    rp0, col0 = random_graph(n, deg, seed=seed)
    s = _split(rp0, col0, 0.25, seed)
    A, H = _dense(n, s.rowptr, s.col), _dense(n, s.ho_rowptr, s.ho_col)
    assert not (A & H).any() and (H == H.T).all() and not H.diagonal().any()
    rng = np.random.default_rng(seed)
    F = 0.05 + 0.45 * rng.random((n, k))
    X = F @ F.T
    assert X.min() > 1e-3 and X.max() < 9.0                                   # p strictly inside (MIN_P_, MAX_P_)
    P = M.make_params(k)
    sumF = F.sum(axis=0)
    off = ~np.eye(n, dtype=bool)
    rest = ~A & ~H & off
    l_mask = 0.5 * (np.log1p(-np.exp(-X[A])).sum() - X[rest].sum())
    v = M.llh(s.rowptr, s.col, s.ho_rowptr, s.ho_col, F, sumF, P)
    assert abs(v - 2.0 * l_mask) <= 1e-12 * abs(2.0 * l_mask)
    r = M.step(s.rowptr, s.col, s.ho_rowptr, s.ho_col, F, sumF, P, early_exit=False, want_pre=True)
    W = np.where(A, np.exp(-X) / (1.0 - np.exp(-X)), 0.0)
    grad = W @ F - rest.astype(float) @ F
    has_nb = A.any(axis=1)
    assert np.abs(r.grad[has_nb] - grad[has_nb]).max() <= 1e-11 * np.abs(grad).max()
    for u in np.nonzero(has_nb)[0]:
        lu = np.log1p(-np.exp(-X[u, A[u]])).sum() - F[u] @ F[rest[u]].sum(axis=0)
        assert abs(r.llh_u[u] - lu) <= 1e-11 * max(abs(lu), 1.0)
    assert (r.accepted[~has_nb] == -1).all()


def test_empty_lists_give_the_bits_of_oracle_step(oracle):
    rp, col = random_graph(300, 8, seed=7, hub=40)
    n, k = len(rp) - 1, 9
    rng = np.random.default_rng(7)
    F = np.where(rng.random((n, k)) < 0.3, rng.random((n, k)), 0.0)
    sumF = oracle.colsum(F)
    P = oracle.make_params(k)
    hr, hc = np.zeros(n + 1, dtype=np.int64), np.zeros(0, dtype=np.int32)
    for mask in (None, (np.arange(n) % 3 == 0).astype(np.uint8)):
        a = oracle.step(rp, col, F, sumF, P, node_mask=mask, want_pre=True)
        b = M.step(rp, col, hr, hc, F, sumF, M.make_params(k), node_mask=mask, want_pre=True)
        assert np.array_equal(a.F, b.F) and np.array_equal(a.sumF, b.sumF) and a.llh == b.llh
        assert np.array_equal(a.accepted, b.accepted) and np.array_equal(a.grad, b.grad) and np.array_equal(a.llh_u, b.llh_u)
    assert oracle.llh(rp, col, F, sumF, P) == M.llh(rp, col, hr, hc, F, sumF, P)
    m1, l1 = oracle.armijo_margins(rp, col, F, sumF, P, np.arange(20))
    m2, l2 = M.armijo_margins(rp, col, hr, hc, F, sumF, P, np.arange(20))
    assert np.array_equal(m1, m2) and np.array_equal(l1, l2)
    r1 = oracle.run(rp, col, F, sumF, P, max_outer=5)
    r2 = M.run(rp, col, hr, hc, F, sumF, P, max_outer=5)
    assert np.array_equal(r1[0], r2[0]) and r1[2] == r2[2] and r1[3] == r2[3] and np.array_equal(r1[4], r2[4])


@pytest.mark.parametrize("seed", [11, 12])
def test_c_oracle_and_numpy_twin_agree(seed):
    rp0, col0 = random_graph(120, 7, seed=seed)
    s = _split(rp0, col0, 0.2, seed)
    n, k = len(rp0) - 1, 6
    rng = np.random.default_rng(seed)
    F = np.where(rng.random((n, k)) < 0.4, rng.random((n, k)), 0.0)
    sumF = F.sum(axis=0)
    P = M.make_params(k)
    for _ in range(3):
        r = M.step(s.rowptr, s.col, s.ho_rowptr, s.ho_col, F, sumF, P)
        Ft, st, lt, acct = M.twin_step(s.rowptr, s.col, s.ho_rowptr, s.ho_col, F, sumF)
        agree = r.accepted == acct
        assert agree.mean() > 0.98, agree.mean()
        # where both accepted the same candidate the rows agree to reassociation noise
        assert np.abs(r.F[agree] - Ft[agree]).max() <= 1e-10 * max(1.0, np.abs(Ft).max())
        if agree.all():
            assert abs(r.llh - lt) <= 1e-10 * abs(lt) and np.allclose(r.sumF, st, rtol=1e-12, atol=1e-10)
        F, sumF = r.F, r.sumF


def test_holdout_llh_is_the_direct_formula():
    rp0, col0 = random_graph(200, 9, seed=5)
    s = _split(rp0, col0, 0.2, 5)
    n, k = len(rp0) - 1, 7
    rng = np.random.default_rng(5)
    F = np.where(rng.random((n, k)) < 0.5, 2.0 * rng.random((n, k)), 0.0)      # some pairs at x = 0 and x > x_hi: both clamps bind
    P = M.make_params(k)
    v, npairs = M.holdout_llh(s.ho_rowptr, s.ho_col, s.ho_is_edge, F, P)
    u = np.repeat(np.arange(n), np.diff(s.ho_rowptr))
    once = u < s.ho_col
    x = np.einsum("ij,ij->i", F[u[once]], F[s.ho_col[once]])
    p = np.clip(np.exp(-x), 1e-4, 0.9999)
    want = np.where(s.ho_is_edge[once] == 1, np.log(1.0 - p), np.log(p)).sum()
    assert npairs == once.sum() == len(s.ho_col) // 2
    assert abs(v - want) <= 1e-12 * abs(want)


def test_split_pairs_contract():
    from bigclam_apachespark_b200 import graphs as G
    rp, col, _ = G.load_npz_graph("facebook_combined")
    n = len(rp) - 1
    s = _split(rp, col, 0.2, 0)
    s2 = _split(rp, col, 0.2, 0)
    assert all(np.array_equal(a, b) for a, b in zip(s, s2))                     # deterministic
    s3 = _split(rp, col, 0.2, 1)
    assert not np.array_equal(s.ho_col, s3.ho_col)
    m = len(col) // 2
    h = int(round(0.2 * m))
    lab = s.ho_is_edge.astype(bool)
    assert lab.sum() == 2 * h and (~lab).sum() == 2 * h                        # exact counts, both directions
    A0, A, H = _dense(n, rp, col), _dense(n, s.rowptr, s.col), _dense(n, s.ho_rowptr, s.ho_col)
    E = np.zeros((n, n), dtype=bool)
    hu = np.repeat(np.arange(n), np.diff(s.ho_rowptr))
    E[hu[lab], s.ho_col[lab]] = True
    assert (H == H.T).all() and not H.diagonal().any() and not (A & H).any()   # symmetric, no self pairs, disjoint from training
    assert (E == E.T).all() and np.array_equal(A | E, A0) and not (A & E).any()  # training u held-out edges = E
    assert not (A0 & H & ~E).any()                                             # held-out non-edges are non-adjacent
    assert H.sum() == len(s.ho_col)                                            # no duplicates
    lt = _dense(n, s.ho_rowptr, s.ho_col).astype(np.int8)
    L = np.zeros((n, n), dtype=np.int8)
    L[hu, s.ho_col] = s.ho_is_edge
    assert (L == L.T).all() and (lt >= L).all()                                # labels symmetric
    # training lists keep the original order of the surviving neighbours
    for u in (0, 107, 1684):
        keep = [v for v in col[rp[u]:rp[u + 1]] if not E[u, v]]
        assert list(s.col[s.rowptr[u]:s.rowptr[u + 1]]) == keep


def test_split_pairs_refuses_non_simple_graphs():
    rp = np.array([0, 2, 3, 4], dtype=np.int64)
    with pytest.raises(ValueError, match="repeated"):
        _split(rp, np.array([1, 1, 0, 0], dtype=np.int32), 0.2, 0)             # 0-1 twice (literal multiplicity)
    with pytest.raises(ValueError, match="self loop"):
        _split(np.array([0, 2, 3, 3], dtype=np.int64), np.array([0, 1, 0], dtype=np.int32), 0.2, 0)
    with pytest.raises(ValueError, match="symmetric"):
        _split(np.array([0, 1, 1, 1], dtype=np.int64), np.array([1], dtype=np.int32), 0.2, 0)
