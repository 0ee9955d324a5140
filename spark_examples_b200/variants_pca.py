"""VariantsPcaDriver -- host-side mirror of the reference's driver class, same method names, argument
meaning and error behaviour (src/main/scala/com/google/cloud/genomics/spark/examples/VariantsPca.scala:36-288),
with the Spark map/reduceByKey similarity build (:182-191) and the MLlib eigen call (:224-227) replaced by the
CUDA path behind include/vpca.h.

    conf = PcaConf(["--synthetic", "2504,1000000"])
    driver = VariantsPcaDriver(conf)
    data = driver.getData
    filtered = [driver.filterDataset(d) for d in data]
    callsRdd = driver.getCallsRdd(filtered)
    simMatrix = driver.getSimilarityMatrix(callsRdd)
    result = driver.computePca(simMatrix)
    driver.emitResult(result)                     # VariantsPca.scala:38-50

Multi-GPU: launch one process per GPU (torchrun); partitions are dealt round-robin to the ranks and the partial
Grams are summed with ONE NCCL all-reduce -- the `reduceByKey(_ + _)` of :190.
"""
from __future__ import annotations

import os
import struct
import sys
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np

from . import dist as vdist
from . import model as vmodel
from . import native
from .conf import PcaConf
from .jformat import jdouble
from .records import Call, CallData, Variant
from .parquet_calls import ParquetSlice
from .variants_common import BedSlice, CallsBatch, JoinedSlice, SyntheticSlice, VariantsCommon, VariantsDataset


# ------------------------------------------------------------------------------------------------------------------
# companion-object functions (VariantsPca.scala:54-78)
# ------------------------------------------------------------------------------------------------------------------
def extractCallInfo(variant: Variant, mapping: Dict[str, int]) -> List[CallData]:
    """VariantsPca.scala:56-60.  hasVariation = any allele index > 0 (a no-call, -1, is not variation); an unknown
    callset id raises KeyError, as `mapping(call.callsetId)` throws NoSuchElementException."""
    out = []
    for call in (variant.calls or ()):                      # variant.calls.getOrElse(Seq())
        has_variation = False
        for allele in call.genotype:                        # foldLeft(false)(_ || _ > 0)
            has_variation = has_variation or allele > 0
        out.append(CallData(has_variation, mapping[call.callsetId]))
    return out


def _fmix64(k: int) -> int:
    k ^= k >> 33
    k = (k * 0xFF51AFD7ED558CCD) & 0xFFFFFFFFFFFFFFFF
    k ^= k >> 33
    k = (k * 0xC4CEB9FE1A85EC53) & 0xFFFFFFFFFFFFFFFF
    k ^= k >> 33
    return k


def _rotl64(x: int, r: int) -> int:
    return ((x << r) | (x >> (64 - r))) & 0xFFFFFFFFFFFFFFFF


def murmur3_128(data: bytes, seed: int = 0) -> str:
    """MurmurHash3_x64_128 -- what Guava's `Hashing.murmur3_128()` computes (un-vendored dependency, shaded at
    build.sbt:44); returns `HashCode.toString`: the 16 bytes (h1 then h2, little-endian) in hex."""
    c1, c2, M = 0x87C37B91114253D5, 0x4CF5AD432745937F, 0xFFFFFFFFFFFFFFFF
    h1 = h2 = seed & M
    n = len(data)
    nblocks = n // 16
    for i in range(nblocks):
        k1, k2 = struct.unpack_from("<QQ", data, i * 16)
        k1 = (k1 * c1) & M; k1 = _rotl64(k1, 31); k1 = (k1 * c2) & M; h1 ^= k1
        h1 = _rotl64(h1, 27); h1 = (h1 + h2) & M; h1 = (h1 * 5 + 0x52DCE729) & M
        k2 = (k2 * c2) & M; k2 = _rotl64(k2, 33); k2 = (k2 * c1) & M; h2 ^= k2
        h2 = _rotl64(h2, 31); h2 = (h2 + h1) & M; h2 = (h2 * 5 + 0x38495AB5) & M
    tail = data[nblocks * 16:]
    k1 = k2 = 0
    t = len(tail)
    if t > 8:
        k2 = int.from_bytes(tail[8:], "little")
        k2 = (k2 * c2) & M; k2 = _rotl64(k2, 33); k2 = (k2 * c1) & M; h2 ^= k2
    if t > 0:
        k1 = int.from_bytes(tail[:8], "little")
        k1 = (k1 * c1) & M; k1 = _rotl64(k1, 31); k1 = (k1 * c2) & M; h1 ^= k1
    h1 ^= n; h2 ^= n
    h1 = (h1 + h2) & M; h2 = (h2 + h1) & M
    h1 = _fmix64(h1); h2 = _fmix64(h2)
    h1 = (h1 + h2) & M; h2 = (h2 + h1) & M
    return (struct.pack("<QQ", h1, h2)).hex()


def variantKeyBytes(variant: Variant, debug: bool = False) -> bytes:
    """The bytes VariantsPca.scala:65-73 feeds the hasher: putString(contig), putLong(start), putLong(end),
    putString(referenceBases), putString(alternateBases.mkString("")) -- Guava writes longs little-endian."""
    alternate = "".join(variant.alternateBases) if variant.alternateBases is not None else ""
    reference = variant.referenceBases if variant.referenceBases is not None else ""
    if debug:
        print(f"{variant.contig}: ({variant.start}, {variant.end}) ref={reference} alt={alternate}")
    return (variant.contig.encode("utf-8") + struct.pack("<q", variant.start) + struct.pack("<q", variant.end) +
            reference.encode("utf-8") + alternate.encode("utf-8"))


def getVariantKey(variant: Variant, debug: bool = False) -> str:
    """VariantsPca.scala:62-78: murmur3_128 of contig, start, end, reference bases, joined alternate bases (host
    restatement; the product path hashes the same bytes on the GPU, vpca_hash_keys / vpca_join_rows)."""
    return murmur3_128(variantKeyBytes(variant, debug))


# ------------------------------------------------------------------------------------------------------------------
# RDD stand-ins
# ------------------------------------------------------------------------------------------------------------------
class CallsRdd:
    """`RDD[Seq[Int]]` (VariantsPca.scala:153): partitions of rows; a row lists the sample indices with variation."""

    def __init__(self, partitions: Sequence[object], n_samples: int):
        self.partitions = list(partitions)       # CallsBatch | SyntheticSlice | BedSlice
        self.n_samples = n_samples

    def collect(self) -> List[List[int]]:
        rows: List[List[int]] = []
        for p in self.partitions:
            if isinstance(p, SyntheticSlice):
                raise RuntimeError("synthetic partitions are generated on the device; use getSimilarityMatrix")
            if isinstance(p, BedSlice):
                from . import plink
                p = CallsBatch(*plink.rows_to_calls(p.rows(), self.n_samples, p.counted))
            if isinstance(p, ParquetSlice):
                p = p.load()
            if isinstance(p, JoinedSlice):
                p = joined_rows_on_host(p)
            for v in range(len(p.offsets) - 1):
                rows.append(p.idx[p.offsets[v]:p.offsets[v + 1]].tolist())
        return rows

    def count(self) -> int:
        return sum(p.nv if isinstance(p, (SyntheticSlice, BedSlice, ParquetSlice)) else len(p.offsets) - 1
                   for p in self.partitions)


class SimilarityMatrix:
    """The `RDD[((Int, Int), Int)]` of VariantsPca.scala:182-191 (all N^2 keys present), resident on the GPU: it
    iterates / collects as ((row, col), count) records like the reference's RDD and additionally remembers the device
    handle, so `computePca` can run on the resident matrix without the N^2 records ever being materialised (the
    Scala twin is `GramRDD`, spark_examples_b200/jvm/GramRDD.scala)."""

    def __init__(self, nat: native.NativePca, n: int):
        self._nat, self.n = nat, n
        self._host: Optional[np.ndarray] = None

    def __iter__(self):
        S = self.toArray()
        for i in range(self.n):
            row = S[i]
            for j in range(self.n):
                yield ((i, j), int(row[j]))

    def toArray(self) -> np.ndarray:
        if self._host is None:
            self._host = self._nat.getGram()
        return self._host

    def collect(self) -> List[Tuple[Tuple[int, int], int]]:
        S = self.toArray()
        return [((i, j), int(S[i, j])) for i in range(self.n) for j in range(self.n)]


# ------------------------------------------------------------------------------------------------------------------
class VariantsPcaDriver:
    """VariantsPca.scala:81-286."""

    def __init__(self, conf: PcaConf, ctx=None, common: Optional[VariantsCommon] = None):
        self.conf = conf
        self.applicationName = type(self).__name__
        self.common = common if common is not None else VariantsCommon(conf, ctx)
        self._rank, self._world = vdist.rank_world()
        self._nat: Optional[native.NativePca] = None
        self._gram_tensor = None
        self._torch_stream = None

    # -- VariantsPca.scala:87 ---------------------------------------------------------------------------------------
    @property
    def getData(self) -> List[VariantsDataset]:
        return self.common.data

    # -- VariantsPca.scala:96-108 -----------------------------------------------------------------------------------
    def filterDataset(self, data: VariantsDataset) -> VariantsDataset:
        if not self.conf.minAlleleFrequency.isDefined:
            return data
        min_af = self.conf.minAlleleFrequency()
        print(f"Min allele frequency {np.float32(min_af)}.")                  # :99 (Float.toString)

        def keep(variant: Variant) -> bool:
            af = variant.info.get("AF")
            if af is None:
                return False                                  # getOrElse(false)
            return np.float32(float(af[0])) >= np.float32(min_af)   # .get(0).toFloat >= minAlleleFrequency

        def fn(part):
            if isinstance(part, (CallsBatch, SyntheticSlice, BedSlice, ParquetSlice)):
                raise ValueError("--min-allele-frequency needs Variant records (INFO field AF)")
            return [v for v in part if keep(v)]
        return data.map_partitions(fn)

    # -- VariantsPca.scala:115-148 ----------------------------------------------------------------------------------
    def joinDatasets(self, datasets: List[VariantsDataset]) -> List[List[CallData]]:
        """2-way join on the variant key (:115-128); calls of both sides concatenated (`related._1 ++ related._2`)."""
        mapping, debug = self.common.indexes, self.conf.debugDatasets()
        sides = []
        for ds in datasets[:2]:
            table: Dict[str, List[List[CallData]]] = {}
            for part in ds.partitions:
                for v in part:
                    table.setdefault(getVariantKey(v, debug), []).append(extractCallInfo(v, mapping))
            sides.append(table)
        out = []
        for key, left in sides[0].items():
            for l in left:                                      # inner join: cartesian product per key
                for r in sides[1].get(key, ()):
                    out.append(l + r)
        return out

    def mergeDatasets(self, datasets: List[VariantsDataset], variantSetCount: int) -> List[List[CallData]]:
        """N-way merge (:136-148): union, group by key, keep keys seen exactly `variantSetCount` times."""
        mapping = self.common.indexes
        groups: Dict[str, List[List[CallData]]] = {}
        for ds in datasets:
            for part in ds.partitions:
                for v in part:
                    groups.setdefault(getVariantKey(v), []).append(extractCallInfo(v, mapping))
        return [[c for calls in g for c in calls] for g in groups.values() if len(g) == variantSetCount]

    def _joined_slice(self, datasets: List[VariantsDataset], variantSetCount: int) -> JoinedSlice:
        """What joinDatasets / mergeDatasets shuffle, laid out for vpca_join_rows: per variant its key bytes (:65-73) and
        the callset indices with variation (:56-60, :164), datasets in order."""
        mapping, debug = self.common.indexes, self.conf.debugDatasets()
        join = variantSetCount == 2
        keys, lens, idx, n_left = [], [], [], 0
        for d, ds in enumerate(datasets[:2] if join else datasets):
            for part in ds.partitions:
                if isinstance(part, (CallsBatch, SyntheticSlice, BedSlice, ParquetSlice)):
                    raise ValueError("joining datasets needs Variant records (the key is made of contig / start / end / bases)")
                for v in part:
                    keys.append(variantKeyBytes(v, debug and join))
                    row = [c.callsetId for c in extractCallInfo(v, mapping) if c.hasVariation]
                    lens.append(len(row))
                    idx.extend(row)
            if d == 0:
                n_left = len(keys)
        off = np.zeros(len(keys) + 1, np.int64)
        np.cumsum(np.asarray(lens, np.int64), out=off[1:])
        return JoinedSlice(native.JOIN if join else native.MERGE, keys, off, np.asarray(idx, np.int32), n_left, variantSetCount)

    # -- VariantsPca.scala:153-168 ----------------------------------------------------------------------------------
    def getCallsRdd(self, data: List[VariantsDataset]) -> CallsRdd:
        n = len(self.common.indexes)
        # conf.variantSetId().size (:154); sources that are not API variant sets count the datasets they hold
        variantSetCount = len(self.conf.variantSetId()) if self.conf.variantSetId.isSupplied else len(data)
        mapping = self.common.indexes
        if variantSetCount == 1:
            parts = []
            for part in data[0].partitions:
                if isinstance(part, (CallsBatch, SyntheticSlice, BedSlice, ParquetSlice)):
                    parts.append(part)                          # already RDD[Seq[Int]] rows (or their packed form)
                else:
                    # a saved model identifies the variants it keeps by their key (model.py)
                    keys = [variantKeyBytes(v) for v in part] if self._model_flags() else None
                    parts.append(_rows_to_batch([extractCallInfo(v, mapping) for v in part], keys))
            return CallsRdd(parts, n)
        # keying, join / merge and the concatenation of the calls run on the GPU and feed the encoder there (csrc/join.cu);
        # joinDatasets / mergeDatasets above stay as the record-level mirror of the reference's public methods
        return CallsRdd([self._joined_slice(data, variantSetCount)], n)

    # -- VariantsPca.scala:182-191 ----------------------------------------------------------------------------------
    def getSimilarityMatrix(self, callsets: CallsRdd) -> SimilarityMatrix:
        """S = sum over variants of x x^T on the GPU: every partition is one `mapPartitions` task (encode + tcgen05
        Gram into a private staging Gram, committed on success); `reduceByKey(_ + _)` across ranks is one all-reduce."""
        nat = self._native(self.common.n_fitted)
        nat.reset()
        done = self._load_checkpoint(nat, callsets)
        for pid, part in enumerate(callsets.partitions):
            if vdist.partition_owner(pid, self._world) != self._rank or pid in done:
                continue
            if isinstance(part, SyntheticSlice):
                self._accumulate_synthetic(nat, part)
                continue
            if isinstance(part, ParquetSlice):
                part = part.load()                              # row group -> CSR rows, no per-record work
            try:
                if isinstance(part, JoinedSlice):
                    nat.joinRows(part.mode, part.keys, part.offsets, part.idx, part.n_left, part.variant_set_count)
                    nat.accumulateJoined(pid)                   # the joined rows never leave the device
                elif isinstance(part, BedSlice):
                    nat.accumulateBed(pid, part.rows(), part.counted)
                else:
                    nat.accumulateCalls(pid, part.offsets, part.idx)
                nat.commit(pid)
            except Exception:
                nat.abort(pid)
                raise
            done.add(pid)
            self._save_checkpoint(nat, callsets, done, every=16)
        self._save_checkpoint(nat, callsets, done, every=1)
        if self._world > 1:
            # every count of the SUMMED matrix must stay a Java Int (VariantsPca.scala:185): bound it before the sum
            total = vdist.allreduce_count(nat.variantCount(), self._gram_tensor.device)
            if total * nat.max_multiplicity ** 2 > 2 ** 31 - 1:
                raise native.VpcaError(native.VPCA_ERR_OVERFLOW, f"{total} variants over all ranks could overflow an "
                                       "int32 similarity count")
            vdist.allreduce_gram(self._gram_tensor)            # VariantsPca.scala:190
        nat.finalizeGram()
        return SimilarityMatrix(nat, self.common.n_fitted)

    def getSimilarityMatrixStream(self, calls: CallsRdd) -> SimilarityMatrix:
        """VariantsPca.scala:262-279 yields the same matrix (its sparse-row quirk is not reproduced, SURVEY.md 2 row 3);
        on the GPU there is one implementation."""
        return self.getSimilarityMatrix(calls)

    # -- VariantsPca.scala:198-231 ----------------------------------------------------------------------------------
    def computePca(self, matrixEntries) -> List[Tuple[str, float, float]]:
        """`matrixEntries`: what getSimilarityMatrix returned (stays on the GPU), or -- the reference's signature,
        `RDD[((Int, Int), Int)]` (:198) -- any iterable of ((row, col), count) records, which are loaded into the GPU
        (absent keys count 0, like the rows `:216-221` never see)."""
        rowCount = self.common.n_fitted
        numPc = self.conf.numPc()
        if numPc < 2:
            # the reference reads array(i + pca.numRows) (:230) and fails for numPc = 1
            raise IndexError("computePca reads the first two principal components; --num-pc must be >= 2")
        if isinstance(matrixEntries, SimilarityMatrix):
            nat = matrixEntries._nat
        else:
            if self.common.n_projected:
                raise ValueError("--projected-callsets needs the similarity matrix getSimilarityMatrix computed")
            S = np.zeros((rowCount, rowCount), np.int32)
            for (i, j), v in matrixEntries:
                S[i, j] = v                                                      # IndexError like Breeze at :216
            nat = self._native(rowCount)
            nat.setGram(S)
        vecs, evals, nonZeroRows = nat.computePca(numPc)
        print(f"Non zero rows in matrix: {nonZeroRows} / {rowCount}.")           # :208
        self.eigenvalues = evals
        self.components = vecs                                                   # all numPc columns (Python twin prints them)
        self._pca_nat = nat
        reverse = self._row_to_callset()                                         # :228
        return [(reverse[i], float(vecs[i, 0]), float(vecs[i, 1])) for i in range(rowCount)]   # :229-230

    def projectPca(self) -> List[Tuple[str, float, float]]:
        """The callsets of --projected-callsets on the first two PCs of the last computePca: (callsetId, pc1, pc2).  Not
        in the reference: Gower's add-a-point formula on the cross counts, centred with the fitted statistics
        (include/vpca.h, DESIGN.md 3.6); projected coordinates are not corrected for their shrinkage towards 0."""
        y = self._pca_nat.projectPca(self.conf.numPc())
        reverse, n = self._row_to_callset(), self.common.n_fitted
        return [(reverse[n + p], float(y[p, 0]), float(y[p, 1])) for p in range(self.common.n_projected)]

    # -- saved model (model.py, DESIGN.md 3.7) ---------------------------------------------------------------------
    def _model_flags(self) -> bool:
        return self.conf.saveModel.isDefined or self.conf.modelPath.isDefined

    def saveModel(self, callsets: CallsRdd) -> vmodel.PcaModel:
        """After computePca: a second pass over the same partitions through the loadings route of each (calls / PLINK
        rows / device panels), then the model file, written atomically.  Prints `Saved model: ...`."""
        nat, k = self._pca_nat, self.conf.numPc()
        vmodel.check_datasets(len(self.getData))
        loadings, carriers, keys = [], [], []
        source = vmodel.source_of(callsets.partitions) or "positional"
        bim_keys = None
        for part in callsets.partitions:
            if isinstance(part, SyntheticSlice):
                import torch
                panel = 8192
                buf = torch.empty(nat.panelBytes(part.nv, panel), dtype=torch.uint8, device=self._gram_tensor.device)
                nat.synthPanelsDevice(part.seed, part.v0, part.nv, 0, buf.data_ptr(), panel)
                L, c = nat.pcaLoadingsPanels(k, buf.data_ptr(), part.nv, panel)
            elif isinstance(part, BedSlice):
                if bim_keys is None:
                    bim_keys = vmodel.plink_keys(part.bed.prefix)
                L, c = nat.pcaLoadingsBed(k, part.rows(), part.counted)
                keys.extend(bim_keys[part.v0:part.v0 + part.nv])
            else:
                if isinstance(part, ParquetSlice):
                    part = part.load()
                L, c = nat.pcaLoadingsCalls(k, part.offsets, part.idx)
                if source == "records":
                    keys.extend(part.keys)
            loadings.append(L)
            carriers.append(c)
        terms = nat.pcaModelTerms(k)
        counted = 0
        if source == "plink":
            counted = {"A1": 1, "A2": 2}[self.conf.bedCountedAllele().upper()]
        m = vmodel.PcaModel(n_fitted=self.common.n_fitted, num_pc=k, loadings=np.concatenate(loadings) if loadings else
                            np.zeros((0, k)), carriers=np.concatenate(carriers) if carriers else np.zeros(0, np.int32),
                            keys=vmodel.hash_keys(nat, keys) if source != "positional" else np.zeros((0, 2), np.uint64),
                            source=source, counted_allele=counted, max_multiplicity=nat.max_multiplicity, **terms)
        vmodel.save(self.conf.saveModel(), m)
        if self._rank == 0:
            print(vmodel.saved_line(m))
        return m

    def scoreWithModel(self, callsets: CallsRdd) -> List[Tuple[str, float, float]]:
        """Every callset of the input on the first two PCs of the saved model of --model-path: one pass over the
        genotypes through the scoring route of each partition, no Gram and no eigensolve.  Prints the matched count."""
        m = vmodel.load(self.conf.modelPath())
        vmodel.check_datasets(len(self.getData))
        k = self.conf.numPc()
        if k < 2:
            raise IndexError("the output reads the first two principal components; --num-pc must be >= 2")
        source = vmodel.source_of(callsets.partitions) or "positional"
        counted = {"A1": 1, "A2": 2}[self.conf.bedCountedAllele().upper()] if source == "plink" else 0
        vmodel.check_study(m, k, source, counted, callsets.count())
        n = len(self.common.indexes)
        device = self.conf.gpuDevice() if self.conf.gpuDevice.isDefined else int(os.environ.get("LOCAL_RANK", "0"))
        dtype = {"int8": native.DTYPE_I8, "i8": native.DTYPE_I8, "bf16": native.DTYPE_BF16}[self.conf.gpuDtype()]
        nat = self._nat = native.NativePca(n, device=device, dtype=dtype, max_multiplicity=m.max_multiplicity, model=m)
        index = vmodel.ModelIndex(m.keys) if m.keyed else None
        bim_keys, v0 = None, 0
        for pid, part in enumerate(callsets.partitions):
            nv = part.nv if isinstance(part, (SyntheticSlice, BedSlice, ParquetSlice)) else len(part.offsets) - 1
            if index is None:
                rows = vmodel.positional_rows(v0, nv)
            elif isinstance(part, BedSlice):
                if bim_keys is None:
                    bim_keys = vmodel.plink_keys(part.bed.prefix)
                rows = index.rows(vmodel.hash_keys(nat, bim_keys[part.v0:part.v0 + part.nv]))
            else:
                rows = index.rows(vmodel.hash_keys(nat, part.keys))
            v0 += nv
            if isinstance(part, SyntheticSlice):
                import torch
                panel = 8192
                buf = torch.empty(nat.panelBytes(part.nv, panel), dtype=torch.uint8, device=f"cuda:{device}")
                nat.synthPanelsDevice(part.seed, part.v0, part.nv, 0, buf.data_ptr(), panel)
                nat.scorePanels(buf.data_ptr(), part.nv, panel, rows)
                nat.synchronize()                               # `buf` must outlive the kernels that read it
                continue
            try:
                if isinstance(part, BedSlice):
                    nat.scoreBed(pid, part.rows(), rows, part.counted)
                else:
                    if isinstance(part, ParquetSlice):
                        part = part.load()
                    nat.scoreCalls(pid, part.offsets, part.idx, rows)
                nat.commit(pid)
            except Exception:
                nat.abort(pid)
                raise
        y, matched = nat.scoreProject(k)
        if self._rank == 0:
            print(vmodel.matched_line(matched, m))
        reverse = {i: cid for cid, i in self.common.indexes.items()}
        return [(reverse[i], float(y[i, 0]), float(y[i, 1])) for i in range(n)]

    def _row_to_callset(self) -> Dict[int, str]:
        rows = self.common.sample_rows
        return {int(rows[i]): cid for cid, i in self.common.indexes.items()}

    # -- VariantsPca.scala:233-246 ----------------------------------------------------------------------------------
    def emitResult(self, result: Sequence[Tuple[str, float, float]], out=None, suffix: str = "-pca.tsv"):
        out = out or sys.stdout
        rows = []
        for callset_id, pc1, pc2 in result:
            dataset = callset_id.split("-")[0]                                   # :235
            rows.append((self.common.names[callset_id], pc1, pc2, dataset))
        if self._rank == 0:
            for name, pc1, pc2, dataset in sorted(rows, key=lambda t: t[0]):     # :238-239
                out.write(f"{name}\t{dataset}\t{jdouble(pc1)}\t{jdouble(pc2)}\n")
            if self.conf.outputPath.isDefined:                                   # :241-245 (saveAsTextFile layout)
                path = self.conf.outputPath() + suffix
                os.makedirs(path, exist_ok=True)
                with open(os.path.join(path, "part-00000"), "w", encoding="utf-8") as fh:
                    for name, pc1, pc2, dataset in rows:
                        fh.write(f"{name}\t{jdouble(pc1)}\t{jdouble(pc2)}\t{dataset}\n")
                open(os.path.join(path, "_SUCCESS"), "w").close()

    def emitProjected(self, projected: Sequence[Tuple[str, float, float]], out=None):
        """The projected samples after the fitted ones: a count line, then the rows in the layout of emitResult (and
        `<output-path>-projected-pca.tsv`)."""
        if self._rank == 0:
            (out or sys.stdout).write(f"Projected samples: {len(projected)}.\n")
        self.emitResult(projected, out, suffix="-projected-pca.tsv")

    def reportIoStats(self):                                                     # :281
        self.common.reportIoStats()
        if self._nat is not None:
            st = self._nat.stats()
            print(f"GPU stats: variants={st['variants_accumulated']} gramLaunches={st['gram_launches']} "
                  f"kernelLaunches={st['kernel_launches']} h2dBytes={st['h2d_bytes']} lastGramMs={st['last_gram_ms']:.3f} "
                  f"lastEigMs={st['last_eig_ms']:.3f}")

    def stop(self):                                                              # :283-285
        if self._nat is not None:
            self._nat.close()
            self._nat = None

    # -- GPU plumbing --------------------------------------------------------------------------------------------
    def _native(self, n: int) -> native.NativePca:
        if self._nat is not None:
            return self._nat
        device = self.conf.gpuDevice() if self.conf.gpuDevice.isDefined else int(os.environ.get("LOCAL_RANK", "0"))
        dtype = {"int8": native.DTYPE_I8, "i8": native.DTYPE_I8, "bf16": native.DTYPE_BF16}[self.conf.gpuDtype()]
        stream = d_gram = 0
        try:
            import torch
            if torch.cuda.is_available():
                torch.cuda.set_device(device)
                self._torch_stream = torch.cuda.Stream(device=device)
                torch.cuda.set_stream(self._torch_stream)
                # projecting runs: (N + M) x N, the cross block below the fitted Gram (one all-reduce moves both)
                self._gram_tensor = torch.zeros((n + self.common.n_projected, n), dtype=torch.int32,
                                                device=f"cuda:{device}")
                stream, d_gram = self._torch_stream.cuda_stream, self._gram_tensor.data_ptr()
        except ImportError:
            pass
        if self._world > 1 and d_gram == 0:
            raise RuntimeError("multi-rank runs need torch with CUDA for the NCCL all-reduce")
        proj = {}
        if self.common.n_projected:
            proj = dict(n_projected=self.common.n_projected, sample_rows=self.common.sample_rows)
        self._nat = native.NativePca(n, device=device, dtype=dtype, num_pc=max(2, self.conf.numPc()), stream=stream,
                                     d_gram=d_gram, **proj)
        return self._nat

    # -- checkpoint / resume (SURVEY 8f-2): the natural checkpoint of this job is the int32 Gram (25 MB at N = 2504)
    #    plus the set of partitions already folded into it -- the counterpart of the reference's --input-path /
    #    --output-path persistence (GenomicsConf.scala:41,46).  One file per rank; partitions are committed atomically,
    #    so a file never holds a half-applied partition.
    def _checkpoint_file(self) -> Optional[str]:
        if not self.conf.checkpointPath.isDefined:
            return None
        return f"{self.conf.checkpointPath()}.rank{self._rank}of{self._world}.npz"

    def _load_checkpoint(self, nat: native.NativePca, callsets: CallsRdd) -> set:
        path = self._checkpoint_file()
        if path is None or not os.path.exists(path):
            return set()
        ck = np.load(path)
        if int(ck["n_samples"]) != callsets.n_samples or int(ck["n_partitions"]) != len(callsets.partitions):
            raise ValueError(f"checkpoint {path} belongs to a different cohort / partitioning")
        n_projected = int(ck["n_projected"]) if "n_projected" in ck.files else 0
        rows = ck["sample_rows"] if "sample_rows" in ck.files else np.arange(callsets.n_samples, dtype=np.int32)
        if n_projected != self.common.n_projected or not np.array_equal(rows, self.common.sample_rows):
            raise ValueError(f"checkpoint {path} was written with other --projected-callsets")
        nat.loadPartialGram(ck["gram"], int(ck["variants"]))
        print(f"Resumed {len(ck['done'])} / {len(callsets.partitions)} partitions from {path}.")
        return set(int(p) for p in ck["done"])

    def _save_checkpoint(self, nat: native.NativePca, callsets: CallsRdd, done: set, every: int):
        path = self._checkpoint_file()
        if path is None or len(done) == 0 or len(done) % every:
            return
        tmp = path + ".tmp.npz"
        gram, variants = nat.partialGram(with_count=True)
        proj = {}
        if self.common.n_projected:
            proj = dict(n_projected=self.common.n_projected, sample_rows=self.common.sample_rows)
        np.savez(tmp, gram=gram, variants=variants, done=np.array(sorted(done), np.int64), n_samples=callsets.n_samples,
                 n_partitions=len(callsets.partitions), **proj)
        os.replace(tmp, path)

    def _accumulate_synthetic(self, nat: native.NativePca, part: SyntheticSlice, panel: int = 8192):
        """Synthetic partitions are born on the device, directly in the panel layout the Gram kernel streams."""
        import torch
        buf = torch.empty(nat.panelBytes(part.nv, panel), dtype=torch.uint8, device=self._gram_tensor.device)
        nat.synthPanelsDevice(part.seed, part.v0, part.nv, 0, buf.data_ptr(), panel)
        nat.accumulatePanels(buf.data_ptr(), part.nv, panel)
        torch.cuda.current_stream().synchronize()      # `buf` must outlive the kernels that read it


def joined_rows_on_host(p: JoinedSlice) -> CallsBatch:
    """The rows vpca_join_rows produces for `p`, computed with Python dicts (CallsRdd.collect and the tests' reference;
    same order: join by left row then right row, merge by first row of the group), empty rows dropped like :166."""
    rows = [p.idx[p.offsets[i]:p.offsets[i + 1]].tolist() for i in range(len(p.keys))]
    hashed = [murmur3_128(k) for k in p.keys]
    out: List[List[int]] = []
    if p.mode == native.JOIN:
        right: Dict[str, List[int]] = {}
        for j in range(p.n_left, len(rows)):
            right.setdefault(hashed[j], []).append(j)
        for i in range(p.n_left):
            for j in right.get(hashed[i], ()):
                out.append(rows[i] + rows[j])
    else:
        groups: Dict[str, List[int]] = {}
        for i, h in enumerate(hashed):
            groups.setdefault(h, []).append(i)
        for members in groups.values():
            if len(members) == p.variant_set_count:
                out.append([c for i in members for c in rows[i]])
    out = [r for r in out if len(r) > 0]
    off = np.zeros(len(out) + 1, np.int64)
    if out:
        off[1:] = np.cumsum([len(r) for r in out])
    return CallsBatch(off, np.asarray([c for r in out for c in r], np.int32))


def _rows_to_batch(rows: Iterable[Sequence[CallData]], keys: Optional[Sequence[bytes]] = None) -> CallsBatch:
    """VariantsPca.scala:164-167: keep calls with variation, drop empty variants, project to the callset index.
    keys (one per row): kept next to the rows that survive."""
    kept, kept_keys = [], []
    for v, calls in enumerate(rows):
        r = [c.callsetId for c in calls if c.hasVariation]
        if len(r) > 0:
            kept.append(r)
            if keys is not None:
                kept_keys.append(keys[v])
    off = np.zeros(len(kept) + 1, np.int64)
    if kept:
        off[1:] = np.cumsum([len(r) for r in kept])
        idx = np.concatenate([np.asarray(r, np.int32) for r in kept])
    else:
        idx = np.zeros(0, np.int32)
    return CallsBatch(off, idx, kept_keys if keys is not None else None)


def main(args: Optional[Sequence[str]] = None):
    """VariantsPcaDriver.main (VariantsPca.scala:38-50)."""
    conf = PcaConf(list(sys.argv[1:] if args is None else args))
    vmodel.check_flags(conf, int(os.environ.get("WORLD_SIZE", "1")))
    if conf.modelPath.isDefined:
        driver = VariantsPcaDriver(conf)
        vmodel.check_datasets(len(driver.getData))
        callsRdd = driver.getCallsRdd([driver.filterDataset(d) for d in driver.getData])
        driver.emitProjected(driver.scoreWithModel(callsRdd))
        driver.reportIoStats()
        driver.stop()
        return
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
        dist.init_process_group("nccl")
    driver = VariantsPcaDriver(conf)
    data = driver.getData
    if conf.saveModel.isDefined:
        vmodel.check_datasets(len(data))
    filtered = [driver.filterDataset(d) for d in data]
    callsRdd = driver.getCallsRdd(filtered)
    simMatrix = driver.getSimilarityMatrix(callsRdd)
    result = driver.computePca(simMatrix)
    driver.emitResult(result)
    if conf.projectedCallsets.isDefined:
        driver.emitProjected(driver.projectPca())
    driver.reportIoStats()
    if conf.saveModel.isDefined:
        driver.saveModel(callsRdd)
    driver.stop()
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
