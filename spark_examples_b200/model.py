"""Saved PCA model: fit once on a reference panel, project every later cohort from the file (DESIGN.md 3.7).

The model holds per-variant loadings L_vc = sum_f x_fv u_fc and carrier counts n_v of the fitted panel, and the k
eigenvalues, a_c = sum_f u_fc, b_c = sum_f (rs_f / N) u_fc and matrixMean of the fit (include/vpca.h, vpca_pca_*).  With
them a study is placed on the fitted axes in one pass over its own genotypes (vpca_score_*): the panel genotypes, its Gram
and the eigensolve are not needed again.  The coordinates equal those of --projected-callsets on the same data up to
rounding; the reference has no projection step, so they are not pinned by it.

This module owns the file layout (one .npz):
    format "vpca-model-1", n_fitted, num_pc, eigenvalues, col_sums, rowsum_dots, matrix_mean (k each / scalars),
    loadings (V x k float64), carriers (V int32), keys (V x 2 uint64, or 0 x 2 for a positional model),
    source ("records" | "plink" | "positional"), counted_allele (PLINK: 1 = A1, 2 = A2; else 0), max_multiplicity.

Variant identity.  Variant records: the reference's getVariantKey bytes (VariantsPca.scala:62-78), MurmurHash3_x64_128 on
the device (vpca_hash_keys).  PLINK: the same bytes built from the .bim record -- contig normalised as in vcf.py,
start = bp - 1, end = start + len(A2), reference = A2, alternate = A1 -- so a panel and a study that follow A2 = REF,
A1 = ALT match across the two formats.  Parquet and synthetic sources have no identities: the model is positional and a
study must present exactly its V variants.
"""
from __future__ import annotations

import os
import struct
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence

import numpy as np

FORMAT = "vpca-model-1"
SOURCES = ("records", "plink", "positional")


@dataclass
class PcaModel:
    n_fitted: int
    num_pc: int
    eigenvalues: np.ndarray     # (k,)
    col_sums: np.ndarray        # (k,)  a
    rowsum_dots: np.ndarray     # (k,)  b
    matrix_mean: float
    loadings: np.ndarray        # (V, k) float64
    carriers: np.ndarray        # (V,) int32
    keys: np.ndarray            # (V, 2) uint64, or (0, 2) for a positional model
    source: str
    counted_allele: int = 0
    max_multiplicity: int = 2

    @property
    def n_variants(self) -> int:
        return int(self.loadings.shape[0])

    @property
    def keyed(self) -> bool:
        return self.source != "positional"


def save(path: str, m: PcaModel) -> None:
    """Writes `path` atomically (a temporary file next to it, then os.replace)."""
    if m.source not in SOURCES:
        raise ValueError(f"model source must be one of {SOURCES}")
    if m.keyed:
        check_unique(m.keys)
    tmp = f"{path}.tmp.{os.getpid()}"
    with open(tmp, "wb") as fh:
        np.savez(fh, format=np.array(FORMAT), n_fitted=np.int64(m.n_fitted), num_pc=np.int64(m.num_pc),
                 eigenvalues=np.asarray(m.eigenvalues, np.float64), col_sums=np.asarray(m.col_sums, np.float64),
                 rowsum_dots=np.asarray(m.rowsum_dots, np.float64), matrix_mean=np.float64(m.matrix_mean),
                 loadings=np.asarray(m.loadings, np.float64), carriers=np.asarray(m.carriers, np.int32),
                 keys=np.asarray(m.keys, np.uint64).reshape(-1, 2), source=np.array(m.source),
                 counted_allele=np.int64(m.counted_allele), max_multiplicity=np.int64(m.max_multiplicity))
    os.replace(tmp, path)


def load(path: str) -> PcaModel:
    with np.load(path, allow_pickle=False) as z:
        fmt = str(z["format"]) if "format" in z.files else "<none>"
        if fmt != FORMAT:
            raise ValueError(f"{path}: unknown model format {fmt!r} (this version reads {FORMAT!r})")
        m = PcaModel(n_fitted=int(z["n_fitted"]), num_pc=int(z["num_pc"]), eigenvalues=z["eigenvalues"],
                     col_sums=z["col_sums"], rowsum_dots=z["rowsum_dots"], matrix_mean=float(z["matrix_mean"]),
                     loadings=z["loadings"], carriers=z["carriers"], keys=z["keys"].reshape(-1, 2), source=str(z["source"]),
                     counted_allele=int(z["counted_allele"]), max_multiplicity=int(z["max_multiplicity"]))
    k = m.num_pc
    if m.source not in SOURCES or m.loadings.shape != (m.n_variants, k) or m.carriers.shape != (m.n_variants,) or \
            any(np.asarray(t).shape != (k,) for t in (m.eigenvalues, m.col_sums, m.rowsum_dots)) or \
            (m.keyed and m.keys.shape != (m.n_variants, 2)):
        raise ValueError(f"{path}: inconsistent model arrays")
    return m


# ---- variant identity ---------------------------------------------------------------------------------------------
def key_bytes(contig: str, start: int, end: int, reference: str, alternate: str) -> bytes:
    """The bytes getVariantKey hashes (VariantsPca.scala:65-73): contig, start and end as little-endian longs, reference
    bases, joined alternate bases."""
    return (contig.encode("utf-8") + struct.pack("<q", start) + struct.pack("<q", end) + reference.encode("utf-8") +
            alternate.encode("utf-8"))


def bim_key_bytes(rec) -> bytes:
    """Key bytes of a .bim record (plink.BimRecord) as the VCF record REF = A2, ALT = A1 at the same position would
    have them (vcf.read_variants): contig normalised ("chr17" -> "17"; names it does not normalise are kept),
    start = bp - 1, end = start + len(A2)."""
    from .vcf import normalize_contig
    contig = normalize_contig(rec.contig) or rec.contig
    start = rec.position - 1
    return key_bytes(contig, start, start + len(rec.a2), rec.a2, rec.a1)


def check_unique(keys: np.ndarray) -> None:
    k = np.ascontiguousarray(keys, np.uint64).reshape(-1, 2)
    if len(k) == 0:
        return
    u, counts = np.unique(k, axis=0, return_counts=True)
    if (counts > 1).any():
        dup = u[np.argmax(counts > 1)]
        raise ValueError(f"refusing to save a keyed model: variant key {struct.pack('<QQ', int(dup[0]), int(dup[1])).hex()} "
                         f"occurs {int(counts.max())} times (variant identities must be unique)")


class ModelIndex:
    """Host dict from variant key to model row."""

    def __init__(self, keys: np.ndarray):
        k = np.ascontiguousarray(keys, np.uint64).reshape(-1, 2)
        self._rows: Dict[bytes, int] = {k[i].tobytes(): i for i in range(len(k))}
        if len(self._rows) != len(k):
            raise ValueError("model keys are not unique")

    def rows(self, study_keys: np.ndarray) -> np.ndarray:
        """model row of every study variant, -1 where the model has none"""
        k = np.ascontiguousarray(study_keys, np.uint64).reshape(-1, 2)
        return np.fromiter((self._rows.get(k[i].tobytes(), -1) for i in range(len(k))), dtype=np.int32, count=len(k))


# ---- flag checks ----------------------------------------------------------------------------------------------------
def check_flags(conf, world: int) -> None:
    """Refuses the combinations --save-model / --model-path do not cover."""
    save_m, score_m = conf.saveModel.isDefined, conf.modelPath.isDefined
    if not (save_m or score_m):
        return
    if score_m:
        for opt, flag in ((conf.saveModel, "--save-model"), (conf.projectedCallsets, "--projected-callsets"),
                          (conf.checkpointPath, "--checkpoint-path")):
            if opt.isDefined:
                raise ValueError(f"--model-path scores a study against a saved model: it cannot be combined with {flag}")
    if world > 1:
        raise ValueError("--save-model and --model-path run on one process and one GPU (WORLD_SIZE must be 1)")
    if conf.variantSetId.isSupplied and len(conf.variantSetId()) > 1:
        raise ValueError("--save-model and --model-path take one variant set (joined datasets are not covered)")


def check_datasets(n_datasets: int) -> None:
    if n_datasets > 1:
        raise ValueError("--save-model and --model-path take one variant set (joined datasets are not covered)")


def check_study(m: PcaModel, num_pc: int, source: str, counted_allele: int, n_variants: int) -> None:
    """Refusals of a scoring run: more PCs than the model has, a PLINK study counting the other allele than a
    PLINK-fitted model, a positional model and a study of another size, a keyed model and a study without identities."""
    if num_pc > m.num_pc:
        raise ValueError(f"--num-pc {num_pc} is above the {m.num_pc} PCs of the model")
    if source == "plink" and m.source == "plink" and counted_allele != m.counted_allele:
        raise ValueError(f"the model was fitted counting allele A{m.counted_allele}; the study counts A{counted_allele}")
    if not m.keyed and n_variants != m.n_variants:
        raise ValueError(f"the model is positional (fitted on a source without variant identities): the study must have "
                         f"exactly its {m.n_variants} variants, it has {n_variants}")
    if m.keyed and source == "positional":
        raise ValueError(f"the model matches variants by identity ({m.source}); the study source has none")


def plink_keys(bed_prefix: str) -> List[bytes]:
    from . import plink
    return [bim_key_bytes(r) for r in plink.read_bim(bed_prefix)]


def hash_keys(nat, keys: Sequence[bytes]) -> np.ndarray:
    """(V, 2) uint64 MurmurHash3_x64_128 of the key bytes, on the GPU of `nat`."""
    if len(keys) == 0:
        return np.zeros((0, 2), np.uint64)
    return nat.hashKeys(list(keys))


def saved_line(m: PcaModel) -> str:
    return f"Saved model: {m.n_variants} variants, {m.num_pc} PCs, {m.n_fitted} fitted samples."


def matched_line(matched: int, m: PcaModel) -> str:
    return f"Model variants matched: {matched} / {m.n_variants}."


def positional_rows(v0: int, nv: int) -> np.ndarray:
    return np.arange(v0, v0 + nv, dtype=np.int32)


def source_of(parts: Sequence[object]) -> Optional[str]:
    """records | plink | positional for the partitions of a CallsRdd (None: nothing to tell)"""
    from .variants_common import BedSlice, CallsBatch
    for p in parts:
        if isinstance(p, BedSlice):
            return "plink"
        if isinstance(p, CallsBatch) and getattr(p, "keys", None) is not None:
            return "records"
        return "positional"
    return None
