"""Projecting contexts on the GPU: the cross block of the (N + M) x N Gram bit-exact against the oracle for every input
route, dtype and row map; compute_pca unchanged by the projected rows; projected coordinates against the numpy
restatement (tests/projection_reference.py) and against the fitted coordinates of the samples they copy; staging; errors; the CLI.

Reference behaviour extended: VariantsPca.scala:182-191 (similarity counts, restricted to projected x fitted pairs) and
:199-223 (the centring, applied to the new rows with the fitted statistics)."""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
from projection_reference import np_project

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
SEED = 20240901


def _nat(n, m, **kw):
    from spark_examples_b200 import native
    return native.NativePca(n, n_projected=m, **kw)


def _interleaved(n, m, rng):
    """sample_rows with the projected samples scattered through the input order."""
    total = n + m
    proj = np.sort(rng.choice(total, size=m, replace=False))
    fitted = np.setdiff1d(np.arange(total), proj)
    rows = np.empty(total, np.int32)
    rows[fitted] = np.arange(n)
    rows[proj] = n + np.arange(m)
    return rows


def _to_csr(X_src):
    """source-order cohort (samples x variants, multiplicities) -> CSR rows of sample indices"""
    rows = [np.repeat(np.arange(X_src.shape[0]), X_src[:, v]).astype(np.int32) for v in range(X_src.shape[1])]
    off = np.zeros(len(rows) + 1, np.int64)
    off[1:] = np.cumsum([len(r) for r in rows])
    return off, (np.concatenate(rows) if rows else np.zeros(0, np.int32))


def _want(X_src, rows, n):
    """(fitted Gram, cross block) of the cohort laid out in context rows"""
    X = np.zeros_like(X_src)
    X[rows] = X_src
    G = X.astype(np.int64) @ X.astype(np.int64).T
    return G[:n, :n].astype(np.int32), G[n:, :n].astype(np.int32)


def _bits(X_src):
    nv, total = X_src.shape[1], X_src.shape[0]
    stride = (total + 7) // 8
    b = np.zeros((nv, stride * 8), np.uint8)
    b[:, :total] = X_src.T > 0
    return np.packbits(b, axis=1, bitorder="little")


def _bed(X_src):
    """carriers of A1 = dosage > 0 (PLINK code 00 hom A1, 10 het, 11 hom A2)"""
    nv, total = X_src.shape[1], X_src.shape[0]
    code = np.where(X_src.T > 0, 0, 3).astype(np.uint8)
    pad = (-total) % 4
    code = np.concatenate([code, np.zeros((nv, pad), np.uint8)], axis=1).reshape(nv, -1, 4)
    return (code[:, :, 0] | (code[:, :, 1] << 2) | (code[:, :, 2] << 4) | (code[:, :, 3] << 6)).astype(np.uint8)


def _run_route(nat, route, X_src, rows):
    import torch
    off, idx = _to_csr(X_src)
    if route == "calls":
        nat.accumulateCalls(0, off, idx)
    elif route == "u16":
        nat.accumulateCalls16(0, off, idx)
    elif route == "bits":
        nat.accumulateBits(0, _bits(X_src))
    elif route == "bed":
        nat.accumulateBed(0, _bed(X_src), 1)
    elif route == "joined":
        from spark_examples_b200 import native
        keys = [f"k{v}".encode() for v in range(X_src.shape[1])]
        nat.joinRows(native.MERGE, keys, off, idx, 0, 1)
        nat.accumulateJoined(0)
    elif route in ("dense", "panels"):
        X = np.zeros_like(X_src)
        X[rows] = X_src                                    # pre-encoded input is taken in row order
        if route == "dense":
            nat.accumulateDense(X.astype(np.int8))
            return
        P = 256
        nv = X.shape[1]
        npan = (nv + P - 1) // P
        pan = np.zeros((npan, X.shape[0], P), np.int8)
        for p in range(npan):
            w = min(P, nv - p * P)
            pan[p, :, :w] = X[:, p * P:p * P + w]
        buf = torch.from_numpy(pan.reshape(-1)).cuda()
        nat.accumulatePanels(buf.data_ptr(), nv, P)
        nat.synchronize()
        return
    nat.commit(0)


@pytest.mark.parametrize("route", ["calls", "u16", "bits", "bed", "dense", "panels", "joined"])
@pytest.mark.parametrize("interleave", [False, True])
def test_cross_block_bit_exact_every_route(route, interleave):
    rng = np.random.default_rng(7)
    n, m, nv = 300, 17, 700
    X_src = (rng.random((n + m, nv)) < 0.3).astype(np.int64)
    rows = _interleaved(n, m, rng) if interleave else np.arange(n + m, dtype=np.int32)
    with _nat(n, m, sample_rows=rows if interleave else None) as nat:
        _run_route(nat, route, X_src, rows)
        nat.finalizeGram()
        S_want, X_want = _want(X_src, rows, n)
        assert np.array_equal(nat.getGram(), S_want)
        assert np.array_equal(nat.crossGram(), X_want)


@pytest.mark.parametrize("dtype", ["int8", "bf16", "e2m1"])
@pytest.mark.parametrize("n,m", [(300, 17), (47, 1)])
@pytest.mark.parametrize("interleave", [False, True])
def test_cross_block_bit_exact_every_dtype(dtype, n, m, interleave):
    from spark_examples_b200 import native
    rng = np.random.default_rng(n + m)
    nv = 1000
    X_src = (rng.random((n + m, nv)) < 0.4).astype(np.int64) * rng.integers(1, 3, (n + m, nv))   # multiplicities 0..2
    rows = _interleaved(n, m, rng) if interleave else np.arange(n + m, dtype=np.int32)
    dt = {"int8": native.DTYPE_I8, "bf16": native.DTYPE_BF16, "e2m1": native.DTYPE_E2M1}[dtype]
    with _nat(n, m, dtype=dt, sample_rows=rows if interleave else None) as nat:
        off, idx = _to_csr(X_src)
        nat.accumulateCalls(3, off, idx)
        nat.commit(3)
        nat.finalizeGram()
        S_want, X_want = _want(X_src, rows, n)
        assert np.array_equal(nat.getGram(), S_want)
        assert np.array_equal(nat.crossGram(), X_want)


@pytest.mark.parametrize("cta_group", ["1", "2"])
def test_full_size_cross_block_bit_exact(monkeypatch, cta_group):
    """N = M = 2504 on a 64 k-variant slice (non-resident stream-K schedule) against an fp32 matmul (exact: counts < 2^24)."""
    import torch
    monkeypatch.setenv("VPCA_CTA_GROUP", cta_group)
    n = m = 2504
    nv = 65536
    g = torch.Generator(device="cuda").manual_seed(11)
    X = (torch.rand((n + m, nv), device="cuda", generator=g) < 0.3).to(torch.int8)
    with _nat(n, m) as nat:
        nat.accumulateDenseDevice(X.data_ptr(), nv, nv)
        nat.finalizeGram()
        S, C = nat.crossGram(), nat.getGram()
    Xf = X.float()
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        want_S = (Xf[:n] @ Xf[:n].T).to(torch.int32).cpu().numpy()
        want_X = (Xf[n:] @ Xf[:n].T).to(torch.int32).cpu().numpy()
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    assert np.array_equal(C, want_S)
    assert np.array_equal(S, want_X)


def _structured(oracle, total, nv):
    return oracle.c_synth_dense(SEED, total, 0, nv, 0).astype(np.int64)        # population structure, binary


@pytest.mark.parametrize("solver", ["lanczos", "direct"])
def test_projection_of_copies_and_against_numpy(oracle, monkeypatch, solver):
    monkeypatch.setenv("VPCA_EIG", solver)
    n, nv, k = 640, 4096, 2
    Xf = _structured(oracle, n, nv)
    rng = np.random.default_rng(3)
    copies = [0, 17, 333, n - 1]
    extra = _structured(oracle, n + 40, nv)[n:]                                 # other samples of the same structure
    X_src = np.concatenate([Xf, Xf[copies], extra])
    m = len(copies) + len(extra)
    rows = _interleaved(n, m, rng)
    X_in = X_src[rows]                                                          # source s holds context row rows[s]
    off, idx = _to_csr(X_in)
    with _nat(n, m, sample_rows=rows) as nat, _nat(n, 0) as plain:
        nat.accumulateCalls(0, off, idx)
        nat.commit(0)
        nat.finalizeGram()
        po, pi = _to_csr(Xf)
        plain.accumulateCalls(0, po, pi)
        plain.commit(0)
        plain.finalizeGram()
        vecs, evals, nz = nat.computePca(k)
        pv, pe, pnz = plain.computePca(k)
        assert np.array_equal(vecs, pv) and np.array_equal(evals, pe) and nz == pnz   # bit-identical fitted PCs
        y = nat.projectPca(k)
        assert np.array_equal(y, nat.projectPca(k))                              # fixed reduction order
        S, X = nat.getGram(), nat.crossGram()
    scale = np.max(np.abs(vecs), axis=0)
    for p, i in enumerate(copies):
        assert np.array_equal(X[p], S[i])
        assert np.all(np.abs(y[p] - vecs[i]) <= 1e-9 * scale)
    _, y_np = np_project(S, X, vecs, evals)
    assert np.all(np.max(np.abs(y - y_np), axis=0) <= 1e-6 * np.max(np.abs(y_np), axis=0))
    assert y.shape == (m, k)


def test_staging_abort_retry_and_partial_round_trip():
    rng = np.random.default_rng(5)
    n, m, nv = 200, 30, 500
    X_src = (rng.random((n + m, nv)) < 0.3).astype(np.int64)
    rows = _interleaved(n, m, rng)
    off, idx = _to_csr(X_src)
    S_want, X_want = _want(X_src, rows, n)
    with _nat(n, m, sample_rows=rows) as nat:
        nat.accumulateCalls(1, off, idx)
        nat.abort(1)                                   # failed task: nothing of it lands
        nat.accumulateCalls(1, off, idx)               # its retry counts once
        nat.commit(1)
        part, cnt = nat.partialGram(with_count=True)
        assert part.shape == (n + m, n) and cnt == nv
        assert np.array_equal(np.tril(part[:n]), np.tril(S_want)) and np.array_equal(part[n:], X_want)
        nat.reset()
        nat.loadPartialGram(part, cnt)
        nat.finalizeGram()
        assert np.array_equal(nat.getGram(), S_want) and np.array_equal(nat.crossGram(), X_want)


def test_errors():
    from spark_examples_b200 import native
    n, m = 64, 8
    with _nat(n, m) as nat:
        with pytest.raises(native.IndexOutOfRange):
            nat.accumulateCalls(-1, np.array([0, 2], np.int64), np.array([1, n + m], np.int32))
        nat.reset()
        X_src = (np.random.default_rng(1).random((n + m, 300)) < 0.3).astype(np.int64)
        nat.accumulateCalls(-1, *_to_csr(X_src))
        nat.finalizeGram()
        with pytest.raises(native.VpcaError) as ei:
            nat.projectPca(2)
        assert ei.value.code == native.VPCA_ERR_STATE
        with pytest.raises(native.VpcaError) as ei:
            nat.setGram(np.zeros((n, n), np.int32))
        assert ei.value.code == native.VPCA_ERR_UNSUPPORTED
        nat.computePca(2)
        with pytest.raises(native.VpcaError) as ei:
            nat.projectPca(3)
        assert ei.value.code == native.VPCA_ERR_BAD_ARG
        with pytest.raises(native.VpcaError) as ei:
            nat.exportIpcHandle()
        assert ei.value.code == native.VPCA_ERR_UNSUPPORTED
    a, b = _nat(n, m), _nat(n, m)
    with pytest.raises(native.VpcaError) as ei:
        native.setPeersLocal([a, b])
    assert ei.value.code == native.VPCA_ERR_UNSUPPORTED
    a.close(), b.close()
    bad = np.arange(n + m, dtype=np.int32)
    bad[3] = 5
    with pytest.raises(native.VpcaError) as ei:
        _nat(n, m, sample_rows=bad)
    assert ei.value.code == native.VPCA_ERR_BAD_ARG
    with pytest.raises(native.VpcaError) as ei:
        _nat(n, m, gram_band=(0, 32))
    assert ei.value.code == native.VPCA_ERR_UNSUPPORTED


def test_exact_cover_is_refused(monkeypatch):
    from spark_examples_b200 import native
    monkeypatch.setenv("VPCA_EXACT_COVER", "1")
    with pytest.raises(native.VpcaError) as ei:
        _nat(64, 8)
    assert ei.value.code == native.VPCA_ERR_UNSUPPORTED


def _cli(args, tmp_path):
    env = dict(os.environ)
    r = subprocess.run([sys.executable, "-m", "spark_examples_b200"] + args, cwd=str(ROOT), env=env, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    return r.stdout.splitlines()


def test_cli_projects_interleaved_plink_samples(oracle, tmp_path):
    from spark_examples_b200 import native, plink
    n_all, nv = 260, 3000
    d = oracle.c_synth_dense(SEED, n_all, 0, nv, 1).astype(np.int64)               # dosage: carriers of A1 = d > 0
    fam = [(f"pop{i % 3}", f"I{i:04d}") for i in range(n_all)]
    proj = sorted(set(range(5, n_all, 13)))
    keep = [i for i in range(n_all) if i not in proj]
    plink.write_fileset(str(tmp_path / "all"), d, fam=fam)
    plink.write_fileset(str(tmp_path / "fit"), d[keep], fam=[fam[i] for i in keep])
    lst = tmp_path / "proj.txt"
    lst.write_text("".join(f"{fam[i][1]}\n" for i in proj))
    out = _cli(["--bed-path", str(tmp_path / "all"), "--projected-callsets", str(lst), "--variants-per-partition", "1024"],
               tmp_path)
    ref = _cli(["--bed-path", str(tmp_path / "fit"), "--variants-per-partition", "1024"], tmp_path)
    cut = out.index(f"Projected samples: {len(proj)}.")
    fitted = [ln for ln in out[:cut] if ln.count("\t") == 3]
    assert fitted == [ln for ln in ref if ln.count("\t") == 3] and len(fitted) == len(keep)
    projected = [ln.split("\t") for ln in out[cut + 1:] if ln.count("\t") == 3]
    assert [p[0] for p in projected] == sorted(fam[i][1] for i in proj)
    # the same coordinates through the ABI
    rows = np.empty(n_all, np.int32)
    rows[keep] = np.arange(len(keep))
    rows[proj] = len(keep) + np.arange(len(proj))
    bed = plink.BedFile(str(tmp_path / "all"), n_samples=n_all)
    with _nat(len(keep), len(proj), sample_rows=rows) as nat:
        for p, v0 in enumerate(range(0, nv, 1024)):
            nat.accumulateBed(p, bed.rows(v0, min(nv, v0 + 1024)), 1)
            nat.commit(p)
        nat.finalizeGram()
        nat.computePca(2)
        y = nat.projectPca(2)
    by_name = {fam[i][1]: y[q] for q, i in enumerate(proj)}
    for name, _, pc1, pc2 in projected:
        assert abs(float(pc1) - by_name[name][0]) <= 1e-12 and abs(float(pc2) - by_name[name][1]) <= 1e-12
