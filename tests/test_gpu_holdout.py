"""GPU tests of the masked objective (bigclam_set_holdout: held-out pairs on the general path of the sparse-row engine)
and of the held-out log-likelihood kernel, against the masked oracle (tests/holdout_oracle).  Same rules as the unmasked
parity tests (tests/test_gpu_parity.py): rows within 1e-9 relative where the accepted step agrees, and every differing
accepted index a proven tie of the oracle's own (masked) Armijo margins."""
import ctypes as C

import numpy as np
import pytest

from conftest import random_graph
from holdout_oracle import masked as M
from test_gpu_parity import RTOL_TIGHT, TIE_TOL

pytestmark = pytest.mark.gpu


def _split(rp, col, frac=0.2, seed=0):
    from bigclam_apachespark_b200.holdout import split_pairs
    return split_pairs(rp, col, frac, seed)


def _solver(rp, col, K, F0, s=None, sumF=None, **kw):
    from bigclam_apachespark_b200 import BigClam
    b = BigClam(record_accepted=True, sparse_rows=True, **kw)
    b.set_graph(rp, col).set_K(K).set_F(F0, sumF=sumF)
    if s is not None:
        b.set_holdout(s.ho_rowptr, s.ho_col, s.ho_is_edge)
    return b


def _check_masked(b, r, llh, inputs, where="", max_flips=0, max_idx_diff=0.02):
    """tests/test_gpu_parity.py::_check_step with the masked margins proving the ties."""
    rp, col, hr, hc, F_in, sumF_in, P = inputs
    F, acc = b.F, b.accepted()
    scale = max(np.abs(r.F).max(), 1e-300)
    row_err = np.abs(F - r.F).max(axis=1)
    flipped = row_err > RTOL_TIGHT * scale
    assert int(flipped.sum()) <= max_flips, f"{where}: {int(flipped.sum())} rows differ (max err {row_err.max():.3e})"
    idx_diff = acc != r.accepted
    assert not (flipped & ~idx_diff).any(), f"{where}: rows differ although the accepted step is the same"
    if idx_diff.any():
        nodes = np.nonzero(idx_diff)[0]
        margins, llh_u = M.armijo_margins(rp, col, hr, hc, np.ascontiguousarray(F_in), sumF_in, P, nodes)
        nsteps = margins.shape[1]
        for i, u in enumerate(nodes):
            a, o = int(acc[u]), int(r.accepted[u])
            j0 = min(a if a >= 0 else nsteps, o if o >= 0 else nsteps)
            tol = TIE_TOL * max(abs(llh_u[i]), 1.0)
            assert abs(margins[i, j0]) <= tol, f"{where}: node {u} gpu {a} oracle {o}: margin {margins[i, j0]:.3e} is not a tie"
            if a >= 0:
                assert margins[i, a] >= -tol, f"{where}: node {u}: accepted candidate {a} fails the oracle's Armijo test"
    assert idx_diff.mean() <= max_idx_diff, where
    if not flipped.any():
        assert np.allclose(b.sumF, r.sumF, rtol=1e-11, atol=1e-9), where
        assert abs(llh - r.llh) <= 1e-10 * abs(r.llh), where


def _steps(b, rp, col, s, F, sumF, K, nsteps, where, mask=None, max_flips=0, max_idx_diff=0.02):
    P = M.make_params(K)
    for it in range(nsteps):
        llh = b.backtrackingLineSearchs(None if mask is None else np.nonzero(mask)[0])
        r = M.step(rp, col, s.ho_rowptr, s.ho_col, F, sumF, P, node_mask=mask)
        _check_masked(b, r, llh, (rp, col, s.ho_rowptr, s.ho_col, F, sumF, P), where=f"{where} it{it}", max_flips=max_flips,
                      max_idx_diff=max_idx_diff)
        F, sumF = b.F, b.sumF
    return F, sumF


def _random_case(n, k, seed, hub=60, frac=0.2):
    rp0, col0 = random_graph(n, 6, seed=seed, hub=hub)
    s = _split(rp0, col0, frac, seed)
    rng = np.random.default_rng(seed)
    F0 = rng.random((n, k)) * (rng.random((n, k)) < min(1.0, 8.0 / k + 0.05))
    return s, F0, F0.sum(axis=0)


@pytest.mark.parametrize("k", [1, 31, 65, 1000])
def test_masked_step_random_graphs(k):
    s, F0, sumF = _random_case(400, k, seed=k)
    b = _solver(s.rowptr, s.col, k, F0, s, sumF=sumF)
    st = b.tile_stats()
    assert st["n_tiles"] == 0 and st["n_split_hubs"] == 0 and st["n_general_nodes"] == 400      # masked routing
    P = M.make_params(k)
    assert abs(b.loglikelihood() - M.llh(s.rowptr, s.col, s.ho_rowptr, s.ho_col, F0, sumF, P)) <= 1e-10 * abs(b.loglikelihood())
    # (at K = 1000 about 3 % of these 400 nodes sit on a tie after the first step; every differing index is proven a tie above)
    _steps(b, s.rowptr, s.col, s, F0, sumF, k, 3, f"masked k={k}", max_flips=1, max_idx_diff=0.02 if k < 1000 else 0.05)
    b.close()


def test_masked_step_uset_mask():
    n, k = 500, 12
    s, F0, sumF = _random_case(n, k, seed=11, hub=0)
    b = _solver(s.rowptr, s.col, k, F0, s, sumF=sumF)
    mask = (np.random.default_rng(11).random(n) < 0.5).astype(np.uint8)
    _steps(b, s.rowptr, s.col, s, F0, sumF, k, 2, "masked uset", mask=mask)
    assert np.array_equal(b.F[mask == 0], F0[mask == 0])
    b.close()


def test_masked_step_nodes_with_only_held_out_pairs():
    """Nodes whose every edge is held out: never updated, but their llh_u carries the held-out x terms."""
    n, k = 300, 8
    rp0, col0 = random_graph(n, 6, seed=21)
    S = np.arange(0, n, 10)
    inS = np.zeros(n, dtype=bool)
    inS[S] = True
    u = np.repeat(np.arange(n), np.diff(rp0))
    touch = inS[u] | inS[col0]
    keep_rp = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.bincount(u[~touch], minlength=n), out=keep_rp[1:])
    keep_col = col0[~touch]
    # held out: every edge touching S (label 1) plus the non-edges (s, s + 1) for s in S (label 0)
    A = np.zeros((n, n), dtype=bool)
    A[u, col0] = True
    a, bb, lab = list(u[touch]), list(col0[touch]), [1] * int(touch.sum())
    for x in S:
        y = (x + 1) % n
        if not A[x, y]:
            a += [x, y]; bb += [y, x]; lab += [0, 0]
    a, bb, lab = np.array(a), np.array(bb), np.array(lab, dtype=np.uint8)
    o = np.lexsort((bb, a))
    hr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.bincount(a, minlength=n), out=hr[1:])
    from bigclam_apachespark_b200.holdout import Split
    s = Split(keep_rp, keep_col.astype(np.int32), hr, bb[o].astype(np.int32), lab[o])
    assert (np.diff(keep_rp)[S] == 0).all() and (np.diff(hr)[S] > 0).all()
    rng = np.random.default_rng(21)
    F0 = rng.random((n, k)) * (rng.random((n, k)) < 0.5)
    sumF = F0.sum(axis=0)
    b = _solver(s.rowptr, s.col, k, F0, s, sumF=sumF)
    P = M.make_params(k)
    want = M.llh(s.rowptr, s.col, s.ho_rowptr, s.ho_col, F0, sumF, P)
    assert abs(b.loglikelihood() - want) <= 1e-10 * abs(want)
    _steps(b, s.rowptr, s.col, s, F0, sumF, k, 2, "only held-out")
    assert np.array_equal(b.F[S], F0[S])
    b.close()


@pytest.mark.parametrize("name,K,density,nsteps", [("facebook_combined", 10, 0.3, 3), ("com-amazon", 200, 0.05, 2)])
def test_masked_step_real_graphs(graphs, name, K, density, nsteps):
    rp0, col0, _ = graphs.load_npz_graph(name)
    s = _split(rp0, col0, 0.2, 0)
    n = len(rp0) - 1
    F0 = graphs.synthetic_F0(n, K, seed=1234, density=density)
    sumF = F0.sum(axis=0)
    b = _solver(s.rowptr, s.col, K, F0, s, sumF=sumF)
    _steps(b, s.rowptr, s.col, s, F0, sumF, K, nsteps, f"masked {name}", max_flips=5)
    b.close()


def test_masked_run_follows_the_oracle_loop():
    n, k = 800, 20
    s, F0, sumF = _random_case(n, k, seed=5, hub=0)
    b = _solver(s.rowptr, s.col, k, F0, s, sumF=sumF)
    llh = b.SGDFindC(max_outer=200)
    _, s_o, llh_o, calls_o, trace_o = M.run(s.rowptr, s.col, s.ho_rowptr, s.ho_col, F0, sumF, M.make_params(k), max_outer=200)
    assert b.last_calls == calls_o
    assert np.allclose(b.last_trace, trace_o, rtol=1e-9, atol=0.0)
    assert abs(llh - llh_o) <= 1e-9 * abs(llh_o)
    assert np.allclose(b.sumF, s_o, rtol=1e-9, atol=1e-9)
    b.close()


def test_holdout_llh_matches_the_oracle():
    n, k = 600, 16
    s, F0, sumF = _random_case(n, k, seed=8)
    b = _solver(s.rowptr, s.col, k, F0, s, sumF=sumF)
    for _ in range(3):
        F = b.F
        want, npairs = M.holdout_llh(s.ho_rowptr, s.ho_col, s.ho_is_edge, F, M.make_params(k))
        got = b.holdout_loglikelihood()
        assert b.last_holdout_pairs == npairs == len(s.ho_col) // 2
        assert abs(got - want) <= 1e-12 * abs(want), (got, want)
        b.backtrackingLineSearchs()
    b.close()


def test_masked_runs_are_bit_identical():
    n, k = 700, 24
    s, F0, sumF = _random_case(n, k, seed=9, hub=120)
    outs = []
    for _ in range(2):
        b = _solver(s.rowptr, s.col, k, F0, s, sumF=sumF)
        llhs = [b.backtrackingLineSearchs() for _ in range(3)]
        outs.append((llhs, b.F, b.sumF, b.holdout_loglikelihood(), b.loglikelihood()))
        b.close()
    (l1, F1, s1, h1, m1), (l2, F2, s2, h2, m2) = outs
    assert l1 == l2 and np.array_equal(F1, F2) and np.array_equal(s1, s2) and h1 == h2 and m1 == m2


def test_clearing_restores_the_unmasked_bits():
    n, k = 700, 24
    s, F0, sumF = _random_case(n, k, seed=10, hub=120)
    a = _solver(s.rowptr, s.col, k, F0, s, sumF=sumF)
    a.clear_holdout()
    c = _solver(s.rowptr, s.col, k, F0, sumF=sumF)
    assert a.tile_stats()["n_tiles"] == c.tile_stats()["n_tiles"] > 0
    for _ in range(3):
        assert a.backtrackingLineSearchs() == c.backtrackingLineSearchs()
    assert np.array_equal(a.F, c.F) and np.array_equal(a.sumF, c.sumF) and np.array_equal(a.accepted(), c.accepted())
    assert a.loglikelihood() == c.loglikelihood()
    a.close()
    c.close()


def test_input_errors_change_nothing():
    from bigclam_apachespark_b200 import BigClam, BigclamError, _lib
    lib = _lib.load()
    n, k = 200, 6
    s, F0, sumF = _random_case(n, k, seed=12, hub=0)
    b = _solver(s.rowptr, s.col, k, F0, sumF=sumF)
    ref = _solver(s.rowptr, s.col, k, F0, sumF=sumF)

    def call(hr, hc, he, ctx=None):
        hr, hc, he = (np.ascontiguousarray(x) for x in (hr, hc, he))
        return lib.bigclam_set_holdout(ctx or b._ctx, hr.ctypes.data, hc.ctypes.data, he.ctypes.data)

    hr, hc, he = s.ho_rowptr, s.ho_col, s.ho_is_edge
    u0, v0 = 0, int(hc[hr[0]])
    j = int(hr[v0] + np.nonzero(hc[hr[v0]:hr[v0 + 1]] == u0)[0][0])          # the mirror of (u0, v0)
    bad = []
    he2 = he.copy(); he2[j] ^= 1; bad.append(("labels", hr, hc, he2))           # asymmetric labels
    hc2 = hc.copy(); hc2[j] = (u0 + 1) if hc[hr[0]] != u0 + 1 else u0 + 2; bad.append(("mirror", hr, hc2, he))   # asymmetric lists
    hc3 = hc.copy(); hc3[hr[0]] = 0; bad.append(("self", hr, hc3, he))         # self pair
    tr_nb = int(s.col[s.rowptr[0]])
    hc4 = hc.copy(); hc4[hr[0]] = tr_nb; bad.append(("training", hr, hc4, he))  # also a training neighbour
    hc5 = hc.copy(); hc5[hr[0]] = n; bad.append(("range", hr, hc5, he))        # out of range
    he6 = he.copy(); he6[0] = 2; bad.append(("0 nor 1", hr, hc, he6))
    hr7 = hr.copy(); hr7[1] = hr[2] + 1; bad.append(("monotone", hr7, hc, he))
    for what, a1, a2, a3 in bad:
        assert call(a1, a2, a3) == _lib.EINVAL, what
    # duplicates: node 0 lists one partner twice (and the partner lists node 0 twice)
    a = np.concatenate([[0, 0, v0, v0], np.repeat(np.arange(n), np.diff(hr))])
    bcol = np.concatenate([[v0, v0, 0, 0], hc])
    lab = np.concatenate([np.ones(4, dtype=np.uint8), he])
    keep = ~((a == 0) & (bcol == v0)) & ~((a == v0) & (bcol == 0))
    keep[:4] = True
    a, bcol, lab = a[keep], bcol[keep], lab[keep]
    o = np.argsort(a, kind="stable")
    hrd = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.bincount(a, minlength=n), out=hrd[1:])
    assert call(hrd, bcol[o].astype(np.int32), lab[o]) == _lib.EINVAL
    assert b"twice" in lib.bigclam_last_error(b._ctx)
    # nothing changed: the same bits as a context that never saw any of it
    for _ in range(2):
        assert b.backtrackingLineSearchs() == ref.backtrackingLineSearchs()
    assert np.array_equal(b.F, ref.F)
    with pytest.raises(BigclamError, match="no held-out pairs"):
        b.holdout_loglikelihood()
    # a masked context keeps its lists when a later call is refused
    b.set_holdout(hr, hc, he)
    h_before = b.holdout_loglikelihood()
    assert call(hr, hc3, he) == _lib.EINVAL
    assert b.holdout_loglikelihood() == h_before and b.tile_stats()["n_tiles"] == 0
    with pytest.raises(BigclamError):
        lib_rc = lib.bigclam_set_owned_range(b._ctx, 0, n // 2)
        _lib.check(lib_rc, b._ctx)
    # unsupported contexts
    dense = BigClam(record_accepted=True)
    dense.set_graph(s.rowptr, s.col).set_K(k).set_F(F0)
    assert call(hr, hc, he, dense._ctx) == _lib.EUNSUPPORTED
    part = _solver(s.rowptr, s.col, k, F0, sumF=sumF)
    assert lib.bigclam_set_owned_range(part._ctx, 0, n // 2) == _lib.OK
    assert call(hr, hc, he, part._ctx) == _lib.EUNSUPPORTED
    peers = _solver(s.rowptr, s.col, k, F0, sumF=sumF)
    handles = (C.c_char * 128)()
    assert lib.bigclam_xchg_export(peers._ctx, 2, 0, handles) == _lib.OK
    assert call(hr, hc, he, peers._ctx) == _lib.EUNSUPPORTED
    for x in (b, ref, dense, part, peers):
        x.close()


def test_select_K_matches_an_oracle_driven_selection(graphs):
    """select_K on facebook against the same selection driven by the masked oracle: same splits, same F0 (the
    solver's own conductance seeding on the training graph), same stop rule."""
    from bigclam_apachespark_b200 import BigClam
    rp, col, _ = graphs.load_npz_graph("facebook_combined")
    Ks, repeats = [5, 10, 20], 2
    b = BigClam()
    b.set_graph(rp, col)
    K_best, rows = b.select_K(Ks=Ks, repeats=repeats, seed=0)
    want = []
    for K in Ks:
        vals, calls = [], []
        for r in range(repeats):
            s = _split(rp, col, 0.2, r)
            t = BigClam(sparse_rows=True)
            t.set_graph(s.rowptr, s.col)
            F0 = t.initNeighborComF(K)
            t.close()
            P = M.make_params(K)
            F, _, _, c, _ = M.run(s.rowptr, s.col, s.ho_rowptr, s.ho_col, F0, F0.sum(axis=0), P)
            vals.append(M.holdout_llh(s.ho_rowptr, s.ho_col, s.ho_is_edge, F, P)[0])
            calls.append(c)
        want.append((K, float(np.mean(vals)), vals, calls))
    print("select_K:", rows, "oracle:", want)
    for (K, mean, vals, calls), (K2, mean2, vals2, calls2) in zip(rows, want):
        assert K == K2 and calls == calls2
        assert np.allclose(vals, vals2, rtol=1e-6, atol=0.0) and abs(mean - mean2) <= 1e-6 * abs(mean2)
    assert K_best == max(want, key=lambda row: (row[1], -row[0]))[0]
    # refit: the full graph at K_best, fitted, ready for extraction
    assert b.K == K_best and b.n == len(rp) - 1 and np.array_equal(b.col, col)
    assert b.last_calls > 0 and b.F.shape == (len(rp) - 1, K_best)
    b.close()


def test_select_K_refuses_multi_gpu():
    from bigclam_apachespark_b200 import BigClam
    b = BigClam(numGPUs=2)
    rp, col = random_graph(50, 4, seed=1)
    b.set_graph(rp, col)
    with pytest.raises(ValueError, match="one GPU"):
        b.select_K(Ks=[2])


def test_cpp_wrappers(tmp_path):
    """include/bigclam_b200.hpp: set_holdout / holdout_loglikelihood once, against the Python binding's numbers."""
    import os
    import subprocess
    from conftest import REPO
    from test_c_host import product_lib
    n, k = 300, 8
    s, F0, sumF = _random_case(n, k, seed=13, hub=0)
    d = tmp_path
    for name, arr in (("rp", s.rowptr), ("col", s.col), ("hr", s.ho_rowptr), ("hc", s.ho_col), ("he", s.ho_is_edge), ("F", F0)):
        arr.tofile(str(d / f"{name}.bin"))
    src = d / "ho.cpp"
    src.write_text(r'''
#include "bigclam_b200.hpp"
#include <cstdio>
#include <fstream>
#include <vector>
template <class T> std::vector<T> rd(const char *p) {
    std::ifstream f(p, std::ios::binary | std::ios::ate); size_t b = f.tellg(); f.seekg(0);
    std::vector<T> v(b / sizeof(T)); f.read(reinterpret_cast<char *>(v.data()), b); return v; }
int main(int argc, char **argv) {
    if (argc < 2) return 2;
    std::string d = argv[1];
    auto rp = rd<int64_t>((d + "/rp.bin").c_str()); auto col = rd<int32_t>((d + "/col.bin").c_str());
    auto hr = rd<int64_t>((d + "/hr.bin").c_str()); auto hc = rd<int32_t>((d + "/hc.bin").c_str());
    auto he = rd<uint8_t>((d + "/he.bin").c_str()); auto F = rd<double>((d + "/F.bin").c_str());
    bigclam::BigClam b(1, 0, true);
    b.set_graph((int64_t)rp.size() - 1, rp.data(), col.data());
    b.set_K(8);
    b.set_F(F);
    b.set_holdout(hr, hc, he);
    int64_t np_ = 0;
    double h0 = b.holdout_loglikelihood(&np_);
    double l = b.backtrackingLineSearchs();
    double h1 = b.holdout_loglikelihood();
    bool threw = false;
    try { std::vector<int32_t> bad(hc); bad[0] = -1; b.set_holdout(hr, bad, he); } catch (const bigclam::Error &) { threw = true; }
    b.set_holdout({}, {}, {});
    double l2 = b.backtrackingLineSearchs();
    std::printf("%.17g %lld %.17g %.17g %d %.17g\n", h0, (long long)np_, l, h1, threw ? 1 : 0, l2);
    return 0;
}
''')
    exe = d / "ho"
    libdir, libname = product_lib()
    cxx = "/usr/bin/g++" if os.access("/usr/bin/g++", os.X_OK) else "g++"
    subprocess.run([cxx, "-std=c++17", "-Wall", "-Wextra", "-Werror", "-O1", "-I", os.path.join(REPO, "include"), str(src), "-o", str(exe),
                    "-L", libdir, f"-l:{libname}", f"-Wl,-rpath,{libdir}"], check=True)
    out = subprocess.run([str(exe), str(d)], capture_output=True, text=True, check=True).stdout.split()
    h0, npairs, l, h1, threw, l2 = float(out[0]), int(out[1]), float(out[2]), float(out[3]), int(out[4]), float(out[5])
    b = _solver(s.rowptr, s.col, k, F0, s)
    assert h0 == b.holdout_loglikelihood() and npairs == len(s.ho_col) // 2
    assert l == b.backtrackingLineSearchs() and h1 == b.holdout_loglikelihood() and threw == 1
    b.clear_holdout()
    assert l2 == b.backtrackingLineSearchs()
    b.close()
