"""Saved PCA model, host side: the per-variant formula equals Gower's formula of --projected-callsets, the model file,
variant keys of VCF and PLINK records, matching a study to model rows, and every refused flag combination (no GPU).

Reference behaviour extended (the reference has no projection step): VariantsPca.scala:62-78 (the variant key),
:182-191 and :199-223 (similarity and centring, expanded over variants)."""
import numpy as np
import pytest
from model_reference import np_model, np_score
from projection_reference import np_project

from oracle import oracle


def _fit(X_fit, k):
    S = X_fit.astype(np.int64) @ X_fit.astype(np.int64).T
    C, _, _ = oracle.np_center(S)
    w, V = np.linalg.eigh(C)
    order = np.argsort(w)[::-1][:k]
    return S, V[:, order], w[order]


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_loadings_formula_equals_gower(seed):
    rng = np.random.default_rng(seed)
    n, m, nv, k = 60, 15, 400, 3
    X = (rng.random((n + m, nv)) < 0.3).astype(np.int64) + (rng.random((n + m, nv)) < 0.05)
    S, U, evals = _fit(X[:n], k)
    model = np_model(S, X[:n], U, evals)
    y = np_score(model, X[n:], np.arange(nv))
    _, y_gower = np_project(S, X[n:] @ X[:n].T, U, evals)
    assert np.all(np.abs(y - y_gower) <= 1e-12 * np.abs(y_gower).max(axis=0))
    # projected copies of fitted samples come out as their rows of u
    y_fit = np_score(model, X[:n], np.arange(nv))
    assert np.allclose(y_fit, U, rtol=0, atol=1e-12)


def _model(nv=5, k=2, source="records", keys=None):
    from spark_examples_b200 import model as vm
    rng = np.random.default_rng(0)
    if keys is None:
        keys = np.arange(2 * nv, dtype=np.uint64).reshape(nv, 2) if source != "positional" else np.zeros((0, 2), np.uint64)
    return vm.PcaModel(n_fitted=10, num_pc=k, eigenvalues=rng.random(k), col_sums=rng.random(k), rowsum_dots=rng.random(k),
                       matrix_mean=0.25, loadings=rng.random((nv, k)), carriers=np.arange(nv, dtype=np.int32), keys=keys,
                       source=source, counted_allele=1 if source == "plink" else 0)


def test_model_file_round_trip(tmp_path):
    from spark_examples_b200 import model as vm
    for source in ("records", "plink", "positional"):
        m = _model(source=source)
        path = str(tmp_path / f"{source}.npz")
        vm.save(path, m)
        got = vm.load(path)
        for f in ("n_fitted", "num_pc", "matrix_mean", "source", "counted_allele", "max_multiplicity"):
            assert getattr(got, f) == getattr(m, f)
        for f in ("eigenvalues", "col_sums", "rowsum_dots", "loadings", "carriers", "keys"):
            assert np.array_equal(getattr(got, f), getattr(m, f)) and getattr(got, f).dtype == np.asarray(getattr(m, f)).dtype
        assert [p.name for p in tmp_path.iterdir() if "tmp" in p.name] == []


def test_unknown_format_refused(tmp_path):
    from spark_examples_b200 import model as vm
    path = str(tmp_path / "m.npz")
    vm.save(path, _model())
    z = dict(np.load(path))
    z["format"] = np.array("vpca-model-99")
    np.savez(path, **z)
    with pytest.raises(ValueError, match="unknown model format"):
        vm.load(path)


def test_duplicate_key_refused(tmp_path):
    from spark_examples_b200 import model as vm
    keys = np.array([[1, 2], [3, 4], [1, 2]], np.uint64)
    with pytest.raises(ValueError, match="occurs 2 times"):
        vm.save(str(tmp_path / "m.npz"), _model(nv=3, keys=keys))


def test_vcf_and_bim_records_give_the_same_key(tmp_path):
    from spark_examples_b200 import model as vm
    from spark_examples_b200 import plink, vcf
    from spark_examples_b200.variants_pca import getVariantKey, murmur3_128, variantKeyBytes
    vcf.write_vcf(str(tmp_path / "a.vcf"), ["s1", "s2"], [
        dict(chrom="chr17", pos=41196312, ref="A", alt=["G"], gts=["0/1", "0/0"]),
        dict(chrom="17", pos=100, ref="AT", alt=["A"], gts=["1/1", "0/0"])])
    recs = list(vcf.read_variants(str(tmp_path / "a.vcf")))
    bims = [plink.BimRecord("chr17", "rs1", 41196312, "G", "A"), plink.BimRecord("17", "rs2", 100, "A", "AT")]
    for rec, bim in zip(recs, bims):
        assert vm.bim_key_bytes(bim) == variantKeyBytes(rec)
        assert murmur3_128(vm.bim_key_bytes(bim)) == getVariantKey(rec)
    assert vm.bim_key_bytes(bims[0]) != vm.bim_key_bytes(bims[1])


def test_model_rows_matching():
    from spark_examples_b200 import model as vm
    keys = np.arange(20, dtype=np.uint64).reshape(10, 2)
    idx = vm.ModelIndex(keys)
    assert np.array_equal(idx.rows(keys[::-1]), np.arange(10)[::-1])                       # reordered
    assert np.array_equal(idx.rows(keys[[1, 5, 7]]), [1, 5, 7])                             # variants missing
    extra = np.concatenate([keys[:3], np.array([[100, 101], [1, 0]], np.uint64), keys[9:]])
    assert np.array_equal(idx.rows(extra), [0, 1, 2, -1, -1, 9])                           # extra variants
    with pytest.raises(ValueError):
        vm.ModelIndex(np.array([[1, 2], [1, 2]], np.uint64))                               # duplicate key


def test_partial_study_restatement_matches_subset():
    """Scoring a study with missing and extra variants equals scoring its matched subset."""
    rng = np.random.default_rng(4)
    n, m, nv, k = 40, 6, 200, 2
    X = (rng.random((n + m, nv)) < 0.3).astype(np.int64)
    S, U, evals = _fit(X[:n], k)
    model = np_model(S, X[:n], U, evals)
    keep = np.sort(rng.choice(nv, size=150, replace=False))[::-1]
    Xs = np.concatenate([X[n:][:, keep], (rng.random((m, 9)) < 0.5).astype(np.int64)], axis=1)
    rows = np.concatenate([keep, -np.ones(9, np.int64)])
    want = np_score(model, X[n:][:, keep], keep)
    assert np.allclose(np_score(model, Xs, rows), want, rtol=0, atol=1e-12 * np.abs(want).max())


def _conf(*args):
    from spark_examples_b200.conf import PcaConf
    return PcaConf(list(args))


@pytest.mark.parametrize("other", [["--save-model", "b.npz"], ["--projected-callsets", "p.txt"],
                                   ["--checkpoint-path", "ck"]])
def test_model_path_refuses_other_flags(other):
    from spark_examples_b200 import model as vm
    with pytest.raises(ValueError, match="cannot be combined"):
        vm.check_flags(_conf("--model-path", "m.npz", *other), 1)


@pytest.mark.parametrize("flag", ["--save-model", "--model-path"])
def test_multi_rank_and_joined_refused(flag):
    from spark_examples_b200 import model as vm
    with pytest.raises(ValueError, match="WORLD_SIZE"):
        vm.check_flags(_conf(flag, "m.npz"), 2)
    with pytest.raises(ValueError, match="one variant set"):
        vm.check_flags(_conf(flag, "m.npz", "--variant-set-id", "a", "b"), 1)
    with pytest.raises(ValueError, match="one variant set"):
        vm.check_datasets(2)
    vm.check_flags(_conf(flag, "m.npz"), 1)


def test_study_refusals():
    from spark_examples_b200 import model as vm
    m = _model(k=2, source="plink")
    with pytest.raises(ValueError, match="above the 2 PCs"):
        vm.check_study(m, 3, "plink", 1, 5)
    with pytest.raises(ValueError, match="counting allele A1"):
        vm.check_study(m, 2, "plink", 2, 5)
    with pytest.raises(ValueError, match="has none"):
        vm.check_study(m, 2, "positional", 0, 5)
    vm.check_study(m, 2, "records", 0, 7)                  # keyed: any study size
    pos = _model(source="positional")
    with pytest.raises(ValueError, match="exactly its 5 variants"):
        vm.check_study(pos, 2, "positional", 0, 4)
    vm.check_study(pos, 2, "positional", 0, 5)


def test_cli_refusals_before_any_work(tmp_path, monkeypatch):
    from spark_examples_b200 import variants_pca
    with pytest.raises(ValueError, match="cannot be combined"):
        variants_pca.main(["--synthetic", "8,100", "--model-path", "m.npz", "--save-model", "b.npz"])
    monkeypatch.setenv("WORLD_SIZE", "2")
    with pytest.raises(ValueError, match="WORLD_SIZE"):
        variants_pca.main(["--synthetic", "8,100", "--save-model", "b.npz"])
    monkeypatch.setenv("WORLD_SIZE", "1")
    bad = tmp_path / "m.npz"
    np.savez(bad, format=np.array("something-else"))
    with pytest.raises(ValueError, match="unknown model format"):
        variants_pca.main(["--synthetic", "8,100", "--model-path", str(bad)])


def test_vcf_batches_keep_the_keys_of_kept_rows():
    from spark_examples_b200.records import CallData
    from spark_examples_b200.variants_pca import _rows_to_batch
    rows = [[CallData(True, 0)], [CallData(False, 1)], [CallData(True, 1), CallData(True, 0)]]
    b = _rows_to_batch(rows, [b"a", b"b", b"c"])
    assert b.keys == [b"a", b"c"] and list(b.offsets) == [0, 1, 3]
    assert _rows_to_batch(rows).keys is None
