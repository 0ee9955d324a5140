"""Flag surface of the reference (Scallop option classes), kept name for name:
src/main/scala/com/google/cloud/genomics/spark/examples/GenomicsConf.scala:31-101.

Scallop derives `--kebab-case` flags from the camelCase vals (README.md:37-40); every option below is an
`Opt` that is called to read it (`conf.numPc()`) and has `.isDefined`, like a ScallopOption.  Options that
only exist here (GPU device/dtype, synthetic cohort) are additive.
"""
from __future__ import annotations

import argparse
import re
from typing import Any, List, Optional, Sequence


class GoogleGenomicsPublicData:
    """SearchVariantsExample.scala:27-31."""
    Platinum_Genomes = "3049512673186936334"
    Thousand_Genomes_Phase_1 = "10473108253681171589"
    Thousand_Genomes_Phase_3 = "4252737135923902652"


class Opt:
    """A parsed ScallopOption: call it for the value; `.isDefined` is true when supplied or defaulted."""

    def __init__(self, name: str, value: Any, supplied: bool):
        self.name, self._value, self.isSupplied = name, value, supplied

    @property
    def isDefined(self) -> bool:
        return self._value is not None

    def __call__(self):
        if self._value is None:
            raise KeyError(f"option --{self.name} is not defined")     # Scallop throws on apply() of an empty option
        return self._value

    @property
    def get(self):
        return self._value

    def __repr__(self):
        return f"Opt({self.name}={self._value!r})"


def _kebab(name: str) -> str:
    return re.sub(r"(?<!^)(?=[A-Z])", "-", name).lower()


class GenomicsConf:
    """GenomicsConf.scala:31-70."""
    DEFAULT_NUMBER_OF_BASES_PER_SHARD = 1000000
    PLATINUM_GENOMES_BRCA1_REFERENCES = "chr17:41196311:41277499"

    def _options(self):
        # (camelCase name, type, default, is_list)
        return [
            ("basesPerPartition", int, self.DEFAULT_NUMBER_OF_BASES_PER_SHARD, False),   # :35
            ("clientSecrets", str, None, False),                                          # :38
            ("inputPath", str, None, False),                                              # :41
            ("numReducePartitions", int, 10, False),                                      # :42
            ("outputPath", str, None, False),                                             # :46
            ("references", str, [self.PLATINUM_GENOMES_BRCA1_REFERENCES], True),         # :47
            ("sparkMaster", str, None, False),                                            # :52
            ("variantSetId", str, [GoogleGenomicsPublicData.Platinum_Genomes], True),    # :54
        ]

    def __init__(self, arguments: Sequence[str] = ()):
        parser = argparse.ArgumentParser(prog=type(self).__name__, allow_abbrev=False)
        specs = self._options()
        for name, typ, default, is_list in specs:
            flag = "--" + _kebab(name)
            if typ is bool:
                parser.add_argument(flag, dest=name, action="store_true", default=None)
            elif is_list:
                parser.add_argument(flag, dest=name, type=typ, nargs="+", default=None)
            else:
                parser.add_argument(flag, dest=name, type=typ, default=None)
        ns = parser.parse_args(list(arguments))
        for name, typ, default, is_list in specs:
            supplied = getattr(ns, name) is not None
            value = getattr(ns, name) if supplied else default
            if typ is bool and value is None:
                value = False
            setattr(self, name, Opt(_kebab(name), value, supplied))

    # GenomicsConf.scala:58-65 builds a SparkContext; here the "context" is the GPU runtime, created by the driver.
    def newSparkContext(self, className: str):
        return None

    def getPartitioner(self, references: str):
        """GenomicsConf.scala:67-69: fixed-width genomic shards (used by the synthetic/offline sources only to
        decide how many variants go into one partition)."""
        return {"references": references, "basesPerPartition": self.basesPerPartition()}


class PcaConf(GenomicsConf):
    """GenomicsConf.scala:76-101."""

    def _options(self):
        return super()._options() + [
            ("allReferences", bool, False, False),        # :77
            ("debugDatasets", bool, False, False),        # :80
            ("minAlleleFrequency", float, None, False),   # :81
            ("numPc", int, 2, False),                     # :85
            # ---- additive, B200 side ----
            ("gpuDevice", int, None, False),              # CUDA ordinal (default: LOCAL_RANK or 0)
            ("gpuDtype", str, "int8", False),             # int8 | bf16 genotype encoding
            ("synthetic", str, None, False),              # "N,V[,seed]": synthetic cohort instead of the retired API
            ("variantsPerPartition", int, 65536, False),  # rows per partition for offline/synthetic sources
            ("checkpointPath", str, None, False),         # save / resume the similarity matrix + partition watermark
            ("vcfPath", str, None, False),                # VCF file(s), comma-separated: one variant set per file
            ("callsParquetPath", str, None, False),       # Parquet file of calls rows (parquet_calls.py): RDD[Seq[Int]] at rest
            ("bedPath", str, None, False),                # PLINK 1 fileset prefix (.bed/.bim/.fam) as the variants source
            ("bedCountedAllele", str, "A1", False),       # which .bim allele is "variation": A1 (PLINK's minor) or A2
            ("projectedCallsets", str, None, False),      # file of callset names (one per line) placed on the PCs of the
                                                          # others instead of being fitted (VariantsPcaDriver.projectPca)
            ("saveModel", str, None, False),              # after computePca: write the per-variant loadings model (model.py)
            ("modelPath", str, None, False),              # score every callset against a saved model: no Gram, no eigensolve
        ]
