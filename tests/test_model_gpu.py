"""Saved PCA model on the GPU: loadings bit-identical across input routes, chunkings and calls, and equal to X_f^T U;
scoring of a study through the model against vpca_project_pca of a projecting context on the same data; determinism of
partitioned scoring; matching of a reordered, partial study; error codes; the CLI round trip.

Reference behaviour extended (the reference has no projection step): VariantsPca.scala:182-191 and :199-223, expanded over
variants (include/vpca.h, DESIGN.md 3.7)."""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
from model_reference import np_model, np_score

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent


def _native():
    from spark_examples_b200 import native
    return native


def _to_csr(X):
    """samples x variants multiplicities -> CSR rows of sample indices"""
    rows = [np.repeat(np.arange(X.shape[0]), X[:, v]).astype(np.int32) for v in range(X.shape[1])]
    off = np.zeros(len(rows) + 1, np.int64)
    off[1:] = np.cumsum([len(r) for r in rows])
    return off, (np.concatenate(rows) if rows else np.zeros(0, np.int32))


def _bed(X):
    """carriers of A1 = cell > 0 (PLINK code 00 hom A1, 11 hom A2)"""
    nv, total = X.shape[1], X.shape[0]
    code = np.where(X.T > 0, 0, 3).astype(np.uint8)
    pad = (-total) % 4
    code = np.concatenate([code, np.zeros((nv, pad), np.uint8)], axis=1).reshape(nv, -1, 4)
    return (code[:, :, 0] | (code[:, :, 1] << 2) | (code[:, :, 2] << 4) | (code[:, :, 3] << 6)).astype(np.uint8)


def _panels(X, P=256):
    import torch
    nv = X.shape[1]
    npan = (nv + P - 1) // P
    pan = np.zeros((npan, X.shape[0], P), np.int8)
    for p in range(npan):
        w = min(P, nv - p * P)
        pan[p, :, :w] = X[:, p * P:p * P + w]
    return torch.from_numpy(pan.reshape(-1)).cuda(), P


def _fit(X_fit, k, **kw):
    """plain context fitted on X_fit (N x V): (nat, vecs, evals, S)"""
    nat = _native().NativePca(X_fit.shape[0], num_pc=max(k, 2), **kw)
    off, idx = _to_csr(X_fit)
    nat.accumulateCalls(0, off, idx)
    nat.commit(0)
    nat.finalizeGram()
    vecs, evals, _ = nat.computePca(k)
    return nat, vecs, evals, nat.getGram()


def _model(nat, X_fit, k):
    off, idx = _to_csr(X_fit)
    L, cnt = nat.pcaLoadingsCalls(k, off, idx)
    terms = nat.pcaModelTerms(k)
    return dict(loadings=L, carriers=cnt, n_fitted=X_fit.shape[0], **terms)


class _M:
    def __init__(self, d):
        self.__dict__.update(d)


@pytest.mark.parametrize("dtype", ["i8", "bf16", "e2m1"])
def test_loadings_bit_identical_across_routes_and_chunks(dtype):
    native = _native()
    dt = {"i8": native.DTYPE_I8, "bf16": native.DTYPE_BF16, "e2m1": native.DTYPE_E2M1}[dtype]
    rng = np.random.default_rng(3)
    n, nv, k = 300, 20000, 4
    X = (rng.random((n, nv)) < 0.2).astype(np.int64)
    nat, vecs, evals, S = _fit(X, k, dtype=dt)
    off, idx = _to_csr(X)
    L, cnt = nat.pcaLoadingsCalls(k, off, idx)
    want = np_model(S, X, vecs, evals)
    assert np.array_equal(cnt, want["carriers"])
    scale = np.abs(want["loadings"]).max(axis=0)
    assert np.all(np.abs(L - want["loadings"]) <= 1e-12 * scale)
    L2, cnt2 = nat.pcaLoadingsCalls(k, off, idx)                        # repeated call
    assert np.array_equal(L2.view(np.int64), L.view(np.int64)) and np.array_equal(cnt2, cnt)
    Lb, cntb = nat.pcaLoadingsBed(k, _bed(X), 1)                        # PLINK rows
    assert np.array_equal(Lb.view(np.int64), L.view(np.int64)) and np.array_equal(cntb, cnt)
    Lh, _ = nat.pcaLoadingsCalls(k, off[:7001], idx[:off[7000]])        # a call that ends mid-chunk
    assert np.array_equal(Lh.view(np.int64), L[:7000].view(np.int64))
    if dtype == "i8":
        buf, P = _panels(X)
        Lp, cntp = nat.pcaLoadingsPanels(k, buf.data_ptr(), nv, P)
        assert np.array_equal(Lp.view(np.int64), L.view(np.int64)) and np.array_equal(cntp, cnt)
    nat.close()
    # other chunk sizes: small CSR chunks and small packed chunks
    nat2, vecs2, _, _ = _fit(X, k, dtype=dt, chunk_variants=8192, chunk_nnz=200000)
    assert np.array_equal(vecs2.view(np.int64), vecs.view(np.int64))
    L3, cnt3 = nat2.pcaLoadingsCalls(k, off, idx)
    L4, _ = nat2.pcaLoadingsBed(k, _bed(X), 1)
    assert np.array_equal(L3.view(np.int64), L.view(np.int64)) and np.array_equal(cnt3, cnt)
    assert np.array_equal(L4.view(np.int64), L.view(np.int64))
    nat2.close()


def test_projecting_fit_context_gives_the_plain_loadings():
    native = _native()
    rng = np.random.default_rng(5)
    n, m, nv, k = 256, 40, 3000, 2
    X_src = (rng.random((n + m, nv)) < 0.25).astype(np.int64)   # source order
    rows = rng.permutation(n + m).astype(np.int32)               # source sample s is context row rows[s]
    X_ctx = np.zeros_like(X_src)
    X_ctx[rows] = X_src
    nat, vecs, evals, S = _fit(X_ctx[:n], k)
    L_plain, c_plain = nat.pcaLoadingsCalls(k, *_to_csr(X_ctx[:n]))
    nat.close()
    off, idx = _to_csr(X_src)
    with native.NativePca(n, n_projected=m, sample_rows=rows) as pj:
        pj.accumulateCalls(0, off, idx)
        pj.commit(0)
        pj.finalizeGram()
        v2, _, _ = pj.computePca(k)
        assert np.array_equal(v2.view(np.int64), vecs.view(np.int64))
        L, c = pj.pcaLoadingsCalls(k, off, idx)
        Lb, _ = pj.pcaLoadingsBed(k, _bed(X_src), 1)
    assert np.array_equal(L.view(np.int64), L_plain.view(np.int64)) and np.array_equal(c, c_plain)
    assert np.array_equal(Lb.view(np.int64), L_plain.view(np.int64))


@pytest.mark.parametrize("n,m,nv", [(300, 60, 4000), (2504, 2504, 3000)])
def test_scoring_matches_project_pca(n, m, nv):
    native = _native()
    rng = np.random.default_rng(11)
    k = 2
    X = (rng.random((n + m, nv)) < 0.3).astype(np.int64)
    off, idx = _to_csr(X)
    with native.NativePca(n, n_projected=m) as pj:
        pj.accumulateCalls(0, off, idx)
        pj.commit(0)
        pj.finalizeGram()
        vecs, evals, _ = pj.computePca(k)
        y_proj = pj.projectPca(k)
        L, cnt = pj.pcaLoadingsCalls(k, off, idx)
        terms = pj.pcaModelTerms(k)
        S = pj.getGram()
    model = dict(loadings=L, carriers=cnt, n_fitted=n, **terms)
    want = np_model(S, X[:n], vecs, evals)
    assert np.array_equal(cnt, want["carriers"])
    assert np.allclose(terms["rowsum_dots"], want["rowsum_dots"], rtol=1e-12, atol=1e-9)
    assert terms["matrix_mean"] == want["matrix_mean"]
    with native.NativePca(m, model=_M(model)) as sc:
        o2, i2 = _to_csr(X[n:])
        sc.scoreCalls(-1, o2, i2, np.arange(nv, dtype=np.int32))
        y, matched = sc.scoreProject(k)
    assert matched == nv
    tol = 1e-9 * np.abs(y_proj).max(axis=0)
    assert np.all(np.abs(y - y_proj) <= tol)
    # projected copies of fitted samples land on their fitted coordinates
    with native.NativePca(8, model=_M(model)) as sc:
        o3, i3 = _to_csr(X[:8])
        sc.scoreCalls(-1, o3, i3, np.arange(nv, dtype=np.int32))
        y8, _ = sc.scoreProject(k)
    assert np.all(np.abs(y8 - vecs[:8]) <= 1e-9)


def test_partitioned_scoring_is_deterministic():
    native = _native()
    rng = np.random.default_rng(13)
    n, m, nv, k = 200, 50, 6000, 3
    X = (rng.random((n + m, nv)) < 0.3).astype(np.int64)
    nat, vecs, evals, S = _fit(X[:n], k)
    model = _M(_model(nat, X[:n], k))
    nat.close()
    cuts = [0, 1000, 2500, 4100, nv]
    Xs = X[n:]

    def run(order, retry=None):
        with native.NativePca(m, model=model) as sc:
            for p in order:
                o, i = _to_csr(Xs[:, cuts[p]:cuts[p + 1]])
                rows = np.arange(cuts[p], cuts[p + 1], dtype=np.int32)
                if p == retry:                                 # a failed attempt, aborted, then the retry
                    sc.scoreCalls(p, o, i, rows)
                    sc.abort(p)
                sc.scoreCalls(p, o, i, rows)
            for p in reversed(order):
                sc.commit(p)
            return sc.scoreProject(k)

    y1, m1 = run([0, 1, 2, 3])
    y2, m2 = run([3, 1, 0, 2])
    y3, m3 = run([2, 0, 3, 1], retry=1)
    assert m1 == m2 == m3 == nv
    assert np.array_equal(y1.view(np.int64), y2.view(np.int64))
    assert np.array_equal(y1.view(np.int64), y3.view(np.int64))
    want = np_score(model.__dict__, Xs, np.arange(nv))
    assert np.all(np.abs(y1 - want) <= 1e-9 * np.abs(want).max(axis=0))


def test_partial_reordered_study_matches_restatement():
    native = _native()
    rng = np.random.default_rng(17)
    n, m, nv, k = 200, 30, 5000, 2
    X = (rng.random((n + m, nv)) < 0.3).astype(np.int64)
    nat, vecs, evals, S = _fit(X[:n], k)
    model = _model(nat, X[:n], k)
    nat.close()
    keep = np.sort(rng.choice(nv, size=nv - nv // 10, replace=False))[::-1]      # 10 % removed, the rest reversed
    Xs = X[n:][:, keep]
    rows = keep.astype(np.int32)
    with native.NativePca(m, model=_M(model)) as sc:
        sc.scoreBed(0, _bed(Xs), rows, 1)
        sc.commit(0)
        y, matched = sc.scoreProject(k)
    assert matched == len(keep)
    want = np_score(model, Xs, rows)
    assert np.all(np.abs(y - want) <= 1e-9 * np.abs(want).max(axis=0))
    # panels route, with unmatched variants (-1) in between
    buf, P = _panels(Xs)
    rows2 = rows.copy()
    rows2[::7] = -1
    with native.NativePca(m, model=_M(model)) as sc:
        sc.scorePanels(buf.data_ptr(), Xs.shape[1], P, rows2)
        y2, matched2 = sc.scoreProject(k)
    assert matched2 == int((rows2 >= 0).sum())
    want2 = np_score(model, Xs, rows2)
    assert np.all(np.abs(y2 - want2) <= 1e-9 * np.abs(want2).max(axis=0))


def test_error_codes():
    native = _native()
    rng = np.random.default_rng(19)
    n, nv, k = 64, 500, 2
    X = (rng.random((n, nv)) < 0.3).astype(np.int64)
    off, idx = _to_csr(X)
    with native.NativePca(n) as nat:
        with pytest.raises(native.VpcaError) as ei:
            nat.pcaLoadingsCalls(k, off, idx)                       # before any computePca
        assert ei.value.code == native.VPCA_ERR_STATE
        nat.accumulateCalls(0, off, idx)
        nat.commit(0)
        nat.finalizeGram()
        nat.computePca(k)
        with pytest.raises(native.VpcaError) as ei:
            nat.pcaLoadingsCalls(k + 1, off, idx)                   # k above the k of computePca
        assert ei.value.code == native.VPCA_ERR_BAD_ARG
        with pytest.raises(native.VpcaError) as ei:
            nat.scoreProject(k)                                     # not a scoring context
        assert ei.value.code == native.VPCA_ERR_UNSUPPORTED
        model = _M(_model(nat, X, k))
    with native.NativePca(10, model=model) as sc:
        o, i = _to_csr(X[:10])
        bad = np.arange(nv, dtype=np.int32)
        bad[3] = nv
        with pytest.raises(native.IndexOutOfRange):
            sc.scoreCalls(0, o, i, bad)
        bad[3] = -2
        with pytest.raises(native.IndexOutOfRange):
            sc.scoreCalls(0, o, i, bad)
        for call in (lambda: sc.accumulateCalls(0, o, i), sc.finalizeGram, sc.getGram, lambda: sc.computePca(2),
                     lambda: sc.projectPca(2), sc.partialGram, sc.gramDevicePtr, sc.gatherGram, sc.peerBarrier,
                     lambda: sc.accumulateBed(0, _bed(X[:10]), 1), lambda: sc.setGram(np.zeros((10, 10), np.int32))):
            with pytest.raises(native.VpcaError) as ei:
                call()
            assert ei.value.code == native.VPCA_ERR_UNSUPPORTED
        with pytest.raises(native.VpcaError) as ei:
            sc.scoreProject(k + 1)
        assert ei.value.code == native.VPCA_ERR_BAD_ARG
        sc.scoreCalls(5, o, i, np.arange(nv, dtype=np.int32))
        with pytest.raises(native.VpcaError) as ei:
            sc.scoreProject(k)                                      # partition 5 is neither committed nor aborted
        assert ei.value.code == native.VPCA_ERR_STATE
        sc.abort(5)
        y, matched = sc.scoreProject(k)
        assert matched == 0 and np.all(np.isfinite(y))


def _cli(args, cwd):
    env = dict(os.environ, PYTHONPATH=str(ROOT))
    return subprocess.run([sys.executable, "-m", "spark_examples_b200"] + args, cwd=cwd, env=env, capture_output=True,
                          text=True, check=True).stdout


def test_cli_plink_save_model_then_score(tmp_path):
    from spark_examples_b200 import plink
    rng = np.random.default_rng(23)
    n, m, nv = 120, 25, 1500
    d = (rng.random((n + m, nv)) < 0.3).astype(np.int64) + (rng.random((n + m, nv)) < 0.1)
    fam = [("fam", f"I{i:04d}") for i in range(n + m)]
    plink.write_fileset(str(tmp_path / "panel"), d, fam)
    study = [f"I{i:04d}" for i in range(n, n + m)]
    (tmp_path / "study.txt").write_text("\n".join(study) + "\n")
    base = ["--bed-path", str(tmp_path / "panel"), "--projected-callsets", str(tmp_path / "study.txt"),
            "--variants-per-partition", "400"]
    out0 = _cli(base + ["--output-path", str(tmp_path / "a")], tmp_path)
    out1 = _cli(base + ["--output-path", str(tmp_path / "b"), "--save-model", str(tmp_path / "m.npz")], tmp_path)
    lines0, lines1 = out0.splitlines(), out1.splitlines()
    strip = [ln for ln in lines1 if not ln.startswith("Saved model:")]
    assert [ln for ln in lines0 if not ln.startswith("GPU stats")] == [ln for ln in strip if not ln.startswith("GPU stats")]
    assert f"Saved model: {nv} variants, 2 PCs, {n} fitted samples." in lines1
    assert (tmp_path / "a-pca.tsv" / "part-00000").read_bytes() == (tmp_path / "b-pca.tsv" / "part-00000").read_bytes()
    # the study alone, variants in reverse order (PLINK keys follow the .bim records)
    ds = d[n:, ::-1]
    plink.write_fileset(str(tmp_path / "study"), ds, fam[n:])
    bim = (tmp_path / "panel.bim").read_text().splitlines()[::-1]
    (tmp_path / "study.bim").write_text("\n".join(bim) + "\n")
    out2 = _cli(["--bed-path", str(tmp_path / "study"), "--model-path", str(tmp_path / "m.npz"),
                 "--output-path", str(tmp_path / "c")], tmp_path)
    assert f"Model variants matched: {nv} / {nv}." in out2.splitlines()
    assert f"Projected samples: {m}." in out2.splitlines()

    def rows(path):
        out = {}
        for ln in (path / "part-00000").read_text().splitlines():
            f = ln.split("\t")
            out[f[0]] = (float(f[1]), float(f[2]))
        return out
    want, got = rows(tmp_path / "b-projected-pca.tsv"), rows(tmp_path / "c-projected-pca.tsv")
    assert set(want) == set(got)
    scale = max(abs(v) for pair in want.values() for v in pair)
    for name in want:
        assert np.allclose(got[name], want[name], rtol=1e-9, atol=1e-9 * scale), name
