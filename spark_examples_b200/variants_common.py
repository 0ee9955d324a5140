"""Ingestion glue -- mirror of the reference's VariantsCommon
(src/main/scala/com/google/cloud/genomics/spark/examples/VariantsCommon.scala:33-81).

The reference resolves callsets and variants through the (retired) Google Genomics API
(VariantsCommon.scala:38-50, rdd/VariantsRDD.scala:187-236).  Ingestion is outside the hot path (SURVEY.md 2
rows 11-12); what the hot path needs from it is kept: `indexes` (callset id -> dense index, in source
order, :44-45), `names` (:46-47) and `data`, a list of datasets of `Variant` records split in partitions.
Sources here: `--input-path` (a JSON-lines stand-in for the saved object file of :53-55), `--synthetic N,V[,seed]`
(device generator, DESIGN.md) or records handed over in memory.

`--projected-callsets FILE` (additive) names callsets that are placed on the principal components of the others
instead of being fitted: `indexes` keeps source order, and `sample_rows` maps every source index to its row of the
GPU context -- fitted callsets first, then the projected ones, each in source order.
"""
from __future__ import annotations

import json
from dataclasses import dataclass
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np

from .conf import PcaConf
from .records import Call, Variant


@dataclass
class CallsBatch:
    """One partition already in `RDD[Seq[Int]]` form (VariantsPca.scala:153-168): CSR rows of sample indices."""
    offsets: np.ndarray   # int64, nv + 1
    idx: np.ndarray       # int32
    keys: Optional[list] = None   # getVariantKey bytes of each row (kept for a saved model, model.py), else None


@dataclass
class JoinedSlice:
    """The rows of several datasets (dataset 0 first) with the bytes of their variant keys, to be joined (2 datasets,
    VariantsPca.scala:115-128) or merged (N datasets, :136-148) on the GPU (vpca_join_rows); `offsets` / `idx` hold the
    calls that pass `_.hasVariation` (:164) as callset indices."""
    mode: int                # native.JOIN | native.MERGE
    keys: list               # bytes per row: contig, start, end, reference bases, alternate bases (:65-73)
    offsets: np.ndarray      # int64, rows + 1
    idx: np.ndarray          # int32
    n_left: int              # JOIN: rows of the left dataset
    variant_set_count: int   # MERGE: group size a key must have (:144)


@dataclass
class SyntheticSlice:
    """Variants [v0, v0 + nv) of the synthetic cohort; materialised on the device, never on the host."""
    seed: int
    v0: int
    nv: int


@dataclass
class BedSlice:
    """Variants [v0, v0 + nv) of a PLINK .bed file (plink.py); the packed rows go to the device as they are on disk."""
    bed: object           # plink.BedFile
    v0: int
    nv: int
    counted: int          # 1: carriers of A1, 2: carriers of A2

    def rows(self) -> np.ndarray:
        return self.bed.rows(self.v0, self.v0 + self.nv)


class VariantsDataset:
    """Stand-in for one `RDD[Variant]`: an ordered list of partitions.  A partition is a list of `Variant`
    records, a `CallsBatch`, a `SyntheticSlice`, a `BedSlice` or a `parquet_calls.ParquetSlice`."""

    def __init__(self, partitions: Sequence[object], variantSetId: str = ""):
        self.partitions = list(partitions)
        self.variantSetId = variantSetId

    def map_partitions(self, fn):
        return VariantsDataset([fn(p) for p in self.partitions], self.variantSetId)

    def __len__(self):
        return len(self.partitions)


class VariantsCommon:
    """VariantsCommon.scala:33.  `indexes`/`names` as at :38-50, `data` as at :52-66."""

    def __init__(self, conf: PcaConf, sc=None, callsets: Optional[Sequence[Tuple[str, str]]] = None,
                 datasets: Optional[Sequence[Sequence[Variant]]] = None):
        self.conf = conf
        self.ioStats: Optional[Dict[str, int]] = None
        per_part = conf.variantsPerPartition()
        if datasets is not None:                                   # records handed over in memory
            if callsets is None:
                raise ValueError("callsets=[(id, name), ...] is required with in-memory datasets")
            self._set_callsets(callsets)
            self.data = [VariantsDataset(_chunk(list(ds), per_part), f"mem-{i}") for i, ds in enumerate(datasets)]
        elif conf.synthetic.isDefined:                             # additive: synthetic cohort
            parts = [int(x) for x in conf.synthetic().split(",")]
            n, v = parts[0], parts[1]
            self.synthetic_seed = parts[2] if len(parts) > 2 else 20240901
            self._set_callsets([(f"synth-{i:06d}", f"S{i:06d}") for i in range(n)])
            slices = [SyntheticSlice(self.synthetic_seed, v0, min(per_part, v - v0)) for v0 in range(0, v, per_part)]
            self.data = [VariantsDataset(slices, "synth")]
        elif conf.vcfPath.isDefined:                               # additive: VCF file(s), one variant set each
            from . import vcf
            paths = [p for p in conf.vcfPath().split(",") if p]
            regions = None
            if conf.references.isSupplied and not conf.allReferences():   # explicit --references only (the BRCA1
                regions = vcf.parse_regions(conf.references())             # default would silently empty other files)
            callsets: List[Tuple[str, str]] = []
            self.data = []
            for path in paths:
                callsets += vcf.read_header(path)[0]
                self.data.append(VariantsDataset(_chunk(list(vcf.read_variants(path, regions)), per_part),
                                                 vcf.dataset_stem(path)))
            self._set_callsets(callsets)
        elif conf.callsParquetPath.isDefined:                      # additive: calls rows at rest, one row group = one partition
            from . import parquet_calls
            pf = parquet_calls.CallsParquet(conf.callsParquetPath())
            self._set_callsets(pf.callsets)
            self.data = [VariantsDataset(pf.slices, "parquet")]
        elif conf.bedPath.isDefined:                               # additive: PLINK fileset on disk
            from . import plink
            counted = {"A1": plink.COUNT_A1, "A2": plink.COUNT_A2}[conf.bedCountedAllele().upper()]
            self._set_callsets(plink.read_fam(conf.bedPath()))
            bed = plink.BedFile(conf.bedPath(), n_samples=len(self.indexes))
            slices = [BedSlice(bed, v0, min(per_part, bed.n_variants - v0), counted)
                      for v0 in range(0, bed.n_variants, per_part)]
            self.data = [VariantsDataset(slices, "bed")]
        elif conf.inputPath.isDefined:                             # VariantsCommon.scala:53-55
            callsets, variants = read_variants_file(conf.inputPath())
            self._set_callsets(callsets)
            self.data = [VariantsDataset(_chunk(variants, per_part), "file")]
        else:
            raise RuntimeError(
                "The Google Genomics API the reference streams from (VariantsCommon.scala:38-66) is retired; "
                "give --vcf-path FILE.vcf[.gz][,...], --bed-path PLINK_PREFIX, --calls-parquet-path FILE, --input-path FILE.jsonl "
                "or --synthetic N,V[,seed]")
        self._set_projection(conf)
        print(f"Matrix size: {len(self.indexes)}.")                 # :48

    def _set_callsets(self, callsets: Sequence[Tuple[str, str]]):
        ids = [c[0] for c in callsets]
        self.indexes: Dict[str, int] = {cid: i for i, cid in enumerate(ids)}      # zipWithIndex.toMap (:44-45)
        if len(self.indexes) != len(ids):
            raise ValueError("duplicate callset id")
        self.names: Dict[str, str] = {c[0]: c[1] for c in callsets}              # :46-47

    def _set_projection(self, conf: PcaConf):
        """`n_projected` and `sample_rows` (source index -> context row) from --projected-callsets."""
        n = len(self.indexes)
        self.n_projected = 0
        self.sample_rows = np.arange(n, dtype=np.int32)
        if not conf.projectedCallsets.isDefined:
            return
        self.n_projected, self.sample_rows = projection_rows(self.names, self.indexes,
                                                             read_projected_names(conf.projectedCallsets()))
        if conf.synthetic.isDefined and not np.array_equal(self.sample_rows, np.arange(n, dtype=np.int32)):
            raise ValueError("--synthetic generates its cohort in row order: only the trailing callsets can be projected")

    @property
    def n_fitted(self) -> int:
        return len(self.indexes) - self.n_projected

    def reportIoStats(self):                                        # :68-73
        if self.ioStats is not None:
            print(self.ioStats)


def read_projected_names(path: str) -> List[str]:
    """One callset name per line (the first output column); blank lines are ignored."""
    with open(path, "r", encoding="utf-8") as fh:
        return [ln.strip() for ln in fh if ln.strip()]


def projection_rows(names: Dict[str, str], indexes: Dict[str, int], projected: Sequence[str]) -> Tuple[int, np.ndarray]:
    """(M, sample_rows): the callsets whose name is listed are projected.  sample_rows[source index] = row of the GPU
    context: fitted callsets get rows 0..N-1 and projected ones N..N+M-1, each group in source order.  A name that
    matches no callset or several, and a list that leaves nothing to fit, are errors."""
    by_name: Dict[str, List[str]] = {}
    for cid, name in names.items():
        by_name.setdefault(name, []).append(cid)
    chosen = set()
    for name in projected:
        ids = by_name.get(name, [])
        if not ids:
            raise ValueError(f"--projected-callsets: no callset is named {name!r}")
        if len(ids) > 1:
            raise ValueError(f"--projected-callsets: {len(ids)} callsets are named {name!r}")
        chosen.add(ids[0])
    total = len(indexes)
    if len(chosen) >= total:
        raise ValueError("--projected-callsets lists every callset: nothing is left to fit")
    order = sorted(indexes.items(), key=lambda kv: kv[1])
    fitted = [i for cid, i in order if cid not in chosen]
    proj = [i for cid, i in order if cid in chosen]
    rows = np.empty(total, dtype=np.int32)
    rows[np.asarray(fitted + proj, dtype=np.int64)] = np.arange(total, dtype=np.int32)
    return len(proj), rows


def _chunk(items: List[object], size: int) -> List[List[object]]:
    size = max(1, int(size))
    return [items[i:i + size] for i in range(0, len(items), size)] or [[]]


def read_variants_file(path: str):
    """JSON lines: first line {"callsets": [{"id": .., "name": ..}, ...]}, then one Variant per line with
    "calls": [{"callsetId": .., "genotype": [..]}, ...] (field names of rdd/VariantsRDD.scala:46-54)."""
    callsets, variants = [], []
    with open(path, "r", encoding="utf-8") as fh:
        for ln, line in enumerate(fh):
            line = line.strip()
            if not line:
                continue
            obj = json.loads(line)
            if ln == 0 and "callsets" in obj:
                callsets = [(c["id"], c.get("name", c["id"])) for c in obj["callsets"]]
                continue
            calls = None
            if obj.get("calls") is not None:
                calls = [Call(c["callsetId"], c.get("callsetName", ""), tuple(c.get("genotype", ())),
                              info=c.get("info", {})) for c in obj["calls"]]
            variants.append(Variant(obj.get("contig", ""), obj.get("id", ""), obj.get("names"), int(obj.get("start", 0)),
                                    int(obj.get("end", 0)), obj.get("referenceBases", ""), obj.get("alternateBases"),
                                    obj.get("info", {}), int(obj.get("created", 0)), obj.get("variantSetId", ""), calls))
    return callsets, variants


def write_variants_file(path: str, callsets: Sequence[Tuple[str, str]], variants: Iterable[Variant]):
    with open(path, "w", encoding="utf-8") as fh:
        fh.write(json.dumps({"callsets": [{"id": c[0], "name": c[1]} for c in callsets]}) + "\n")
        for v in variants:
            calls = None
            if v.calls is not None:
                calls = [{"callsetId": c.callsetId, "callsetName": c.callsetName, "genotype": list(c.genotype)}
                         for c in v.calls]
            fh.write(json.dumps({"contig": v.contig, "id": v.id, "start": v.start, "end": v.end,
                                 "referenceBases": v.referenceBases, "alternateBases": v.alternateBases,
                                 "info": v.info, "variantSetId": v.variantSetId, "calls": calls}) + "\n")
