"""Projection of held-out samples onto the fitted PCs, on the CPU: the tile lists of projecting contexts (every needed
cell of the (N + M) x N buffer flushed exactly once), the numpy restatement of the projection formula, and the host
plumbing of --projected-callsets (row map, errors, checkpoint guard, output layouts)."""
import io

import numpy as np
import pytest

import spark_examples_b200 as pkg
from spark_examples_b200 import native
from spark_examples_b200.variants_common import projection_rows
from spark_examples_b200.variants_pca import VariantsPcaDriver
from projection_reference import np_project


def _flush_counts(tiles, n_fit, n_total, cg):
    """Model of the epilogue: tile t writes S[row][col] for B row `row` and A row `col` of either CTA when
    row < min(n_total, rowB + n_eff), col < n_fit and row >= col (rectangle tiling: no transposed blocks, no fillers)."""
    cnt = np.zeros((n_total, n_fit), np.int32)
    row = np.arange(n_total)[:, None]
    for t in tiles:
        rowA0, rowA1, rowB, n_eff, _, flags, acc_cols, _ = (int(x) for x in t)
        assert flags & 3 == 0 and n_eff % 16 == 0 and 0 < n_eff <= acc_cols
        r0, r1 = rowB, min(n_total, rowB + n_eff)
        for a in ([rowA0, rowA1] if cg == 2 else [rowA0]):
            c0, c1 = a, min(n_fit, a + 128)
            if c0 >= c1 or r0 >= r1:
                continue
            col = np.arange(c0, c1)[None, :]
            keep = row[r0:r1] >= col
            cnt[r0:r1, c0:c1] += keep
    return cnt


@pytest.mark.parametrize("mxf4", [False, True])
@pytest.mark.parametrize("cg", [1, 2])
@pytest.mark.parametrize("m", [1, 15, 17, 256, 2504])
@pytest.mark.parametrize("n", [1, 47, 128, 300, 2504])
def test_projection_tiles_flush_every_needed_cell_once(n, m, cg, mxf4):
    tiles = native.debugProjectionTiles(n, n + m, cg, mxf4)
    assert len(tiles) > 0
    # B strips: inside the (N + M)-row buffer, contiguous, starting at 0; A blocks: over [0, N) only
    assert tiles[:, 2].min() == 0 and tiles[:, 2].max() < n + m and tiles[:, 0].max() < n
    cnt = _flush_counts(tiles, n, n + m, cg)
    need = np.tril(np.ones((n + m, n), bool))                       # row >= col, col < N
    assert np.array_equal(cnt, need.astype(np.int32))


@pytest.mark.parametrize("cg", [1, 2])
@pytest.mark.parametrize("n", [2, 47, 128, 300, 2504])
def test_projection_tiles_without_projected_rows_are_the_plain_lists(n, cg):
    assert np.array_equal(native.debugProjectionTiles(n, n, cg, False), native.debugBandTiles(n, cg, 0, n))
    assert np.array_equal(native.debugProjectionTiles(n, n, cg, True), native.debugTiles(n, cg, exact=False))


def _cohort(rng, n, nv, p=0.3):
    return (rng.random((n, nv)) < p).astype(np.int64)


@pytest.mark.parametrize("n,m,k", [(40, 6, 2), (97, 13, 4)])
def test_projection_formula_places_copies_on_their_fitted_rows(oracle, n, m, k):
    rng = np.random.default_rng(n)
    Xf = _cohort(rng, n, 300)
    copies = [0, 5, n - 1]
    Xp = np.concatenate([Xf[copies], _cohort(rng, m - len(copies), 300)])
    S = oracle.np_similarity_dense(Xf)
    X = (Xp @ Xf.T).astype(np.int32)
    C, _, _ = oracle.np_center(S)
    w, V = np.linalg.eigh(C)
    order = np.argsort(w)[::-1][:k]
    U, lam = oracle.sign_normalise(V[:, order]), w[order]
    Cx, Y = np_project(S, X, U, lam)
    for p, i in enumerate(copies):
        assert np.array_equal(X[p], S[i])
        assert np.array_equal(Cx[p], C[i])                          # bit for bit: same centring, same order
        assert np.max(np.abs(Y[p] - U[i])) <= 1e-12 * np.max(np.abs(U))
    # the formula is linear in the centred row: projecting the fitted rows reproduces U (C U = U diag(lam))
    _, Yf = np_project(S, S, U, lam)
    assert np.allclose(Yf, U, atol=1e-12)


# ---- --projected-callsets ------------------------------------------------------------------------------------------
def _names(ids):
    return {cid: cid.split("-")[1] for cid in ids}


def test_sample_rows_put_fitted_callsets_first_in_source_order():
    ids = [f"fam-I{i}" for i in range(7)]
    indexes = {cid: i for i, cid in enumerate(ids)}
    m, rows = projection_rows(_names(ids), indexes, ["I1", "I4", "I5"])
    assert m == 3
    # fitted I0 I2 I3 I6 -> rows 0..3; projected I1 I4 I5 -> rows 4..6
    assert rows.tolist() == [0, 4, 1, 2, 5, 6, 3]
    m, rows = projection_rows(_names(ids), indexes, ["I6"])
    assert m == 1 and rows.tolist() == list(range(7))


def test_projected_names_that_do_not_resolve_are_errors():
    ids = ["a-X", "b-X", "c-Y", "d-Z"]
    indexes = {cid: i for i, cid in enumerate(ids)}
    with pytest.raises(ValueError, match="no callset is named 'Q'"):
        projection_rows(_names(ids), indexes, ["Q"])
    with pytest.raises(ValueError, match="2 callsets are named 'X'"):
        projection_rows(_names(ids), indexes, ["X"])
    with pytest.raises(ValueError, match="nothing is left to fit"):
        projection_rows({"a-X": "X", "c-Y": "Y"}, {"a-X": 0, "c-Y": 1}, ["X", "Y"])


def test_flag_is_parsed_and_read(tmp_path):
    from spark_examples_b200 import plink
    lst = tmp_path / "proj.txt"
    lst.write_text("I002\n\nI000\n")
    d = np.zeros((5, 8), np.int64)
    plink.write_fileset(str(tmp_path / "c"), d, fam=[("f", f"I{i:03d}") for i in range(5)])
    conf = pkg.PcaConf(["--bed-path", str(tmp_path / "c"), "--projected-callsets", str(lst)])
    assert conf.projectedCallsets() == str(lst)
    common = pkg.variants_common.VariantsCommon(conf)
    assert common.n_projected == 2 and common.n_fitted == 3
    assert common.sample_rows.tolist() == [3, 0, 4, 1, 2]
    plain = pkg.variants_common.VariantsCommon(pkg.PcaConf(["--bed-path", str(tmp_path / "c")]))
    assert plain.n_projected == 0 and plain.sample_rows.tolist() == list(range(5))


def test_synthetic_cohort_projects_trailing_callsets_only(tmp_path):
    lst = tmp_path / "p.txt"
    lst.write_text("S000005\nS000004\n")
    common = pkg.variants_common.VariantsCommon(pkg.PcaConf(["--synthetic", "6,1000", "--projected-callsets", str(lst)]))
    assert common.n_projected == 2 and common.sample_rows.tolist() == list(range(6))
    lst.write_text("S000001\n")
    with pytest.raises(ValueError, match="only the trailing callsets"):
        pkg.variants_common.VariantsCommon(pkg.PcaConf(["--synthetic", "6,1000", "--projected-callsets", str(lst)]))


def test_checkpoint_of_another_projection_is_refused(tmp_path):
    from spark_examples_b200 import plink
    plink.write_fileset(str(tmp_path / "c"), np.zeros((6, 10), np.int64), fam=[("f", f"I{i}") for i in range(6)])
    lst = tmp_path / "p.txt"
    lst.write_text("I1\n")
    ck = str(tmp_path / "ck")
    argv = ["--bed-path", str(tmp_path / "c"), "--checkpoint-path", ck]
    driver = VariantsPcaDriver(pkg.PcaConf(argv + ["--projected-callsets", str(lst)]))
    calls = driver.getCallsRdd(driver.getData)
    path = driver._checkpoint_file()
    gram = np.zeros((6, 5), np.int32)
    # written without projection: refused by the projecting run
    np.savez(path, gram=gram, variants=0, done=np.array([0], np.int64), n_samples=6, n_partitions=len(calls.partitions))
    with pytest.raises(ValueError, match="other --projected-callsets"):
        driver._load_checkpoint(None, calls)
    # written with another projected callset
    np.savez(path, gram=gram, variants=0, done=np.array([0], np.int64), n_samples=6, n_partitions=len(calls.partitions),
             n_projected=1, sample_rows=np.array([0, 1, 5, 2, 3, 4], np.int32))
    with pytest.raises(ValueError, match="other --projected-callsets"):
        driver._load_checkpoint(None, calls)
    # and a projecting checkpoint is refused by a plain run
    plain = VariantsPcaDriver(pkg.PcaConf(argv))
    with pytest.raises(ValueError, match="other --projected-callsets"):
        plain._load_checkpoint(None, plain.getCallsRdd(plain.getData))


def test_projected_rows_are_emitted_after_the_fitted_ones(tmp_path):
    from spark_examples_b200 import plink
    plink.write_fileset(str(tmp_path / "c"), np.zeros((4, 8), np.int64), fam=[("fa", "I0"), ("fb", "I1"), ("fa", "I2"),
                                                                              ("fb", "I3")])
    lst = tmp_path / "p.txt"
    lst.write_text("I3\nI1\n")
    out_path = str(tmp_path / "out")
    driver = VariantsPcaDriver(pkg.PcaConf(["--bed-path", str(tmp_path / "c"), "--projected-callsets", str(lst),
                                            "--output-path", out_path]))
    buf = io.StringIO()
    driver.emitResult([("fa-I2", 0.5, -0.25), ("fa-I0", -0.5, 0.25)], buf)
    driver.emitProjected([("fb-I3", 0.125, 1.0), ("fb-I1", -1.0, 0.0)], buf)
    assert buf.getvalue().splitlines() == [
        "I0\tfa\t-0.5\t0.25", "I2\tfa\t0.5\t-0.25", "Projected samples: 2.", "I1\tfb\t-1.0\t0.0", "I3\tfb\t0.125\t1.0"]
    fitted = (tmp_path / "out-pca.tsv" / "part-00000").read_text().splitlines()
    projected = (tmp_path / "out-projected-pca.tsv" / "part-00000").read_text().splitlines()
    assert fitted == ["I2\t0.5\t-0.25\tfa", "I0\t-0.5\t0.25\tfa"]
    assert projected == ["I3\t0.125\t1.0\tfb", "I1\t-1.0\t0.0\tfb"]
    assert (tmp_path / "out-projected-pca.tsv" / "_SUCCESS").exists()
