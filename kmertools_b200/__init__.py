"""kmertools_b200 — B200-native oligonucleotide frequency vectors (one hot path of kmertools).

Layout: csrc/ holds the CUDA kernels and the C ABI (include/kmertools_b200.h); oligo.py and kmers.py mirror
the reference's OligoComputer / KmerGenerator interfaces on top of that ABI.  The top-level `pykmertools` package re-exports
it under the reference's module name.
"""
from .oligo import OligoComputer, MultiOligoComputer, HostBuffer, shard_bounds  # noqa: F401
from .kmers import KmerGenerator, kmer_pairs  # noqa: F401
from .sparse import kmer_counts, kmer_counts_tensors  # noqa: F401
from .counter import KmerCounter  # noqa: F401
from ._lib import KtbError  # noqa: F401

__version__ = "0.1.0"
