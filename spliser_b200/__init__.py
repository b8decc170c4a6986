"""spliser_b200 -- B200-native counting path of SpliSER v0.1.8 (`process` and the `combine` re-count).

The product is libspliser_b200.so (CUDA, sm_100a) behind the C ABI of include/spliser_b200.h; this
package is its Python host side: ctypes binding, numpy API, BED12 parsing, gene assignment, the
SpliSER-compatible CLI and TSV writers.  Importing the package does not need a GPU; creating a
Context does, and there is no CPU fallback.
"""
from .api import (CompactRecords, Context, Junctions, PackedRecords, Records, SiteTable, SpliserError, mode_flags,  # noqa: F401
                  FLAG_COMBINE, FLAG_CRYPTIC, FLAG_RF, FLAG_STRANDED, bam_reference_names)

__version__ = "0.1.0"
