"""sage_b200 — B200-native (sm_100a) fragment-index search-and-score, a drop-in for sage-core's
`IndexedDatabase::query` + `Scorer::score` hot path (lazear/sage). The product is the CUDA library behind the C ABI
in include/sage_b200.h; this package is the thin Python binding used by the tests and the benchmark."""
from .api import (DA, PCT, PPM, Feature, IndexedDatabase, Peptides, Precursor, ProcessedSpectrum, Scorer, SpectraBatch, SpectrumProcessor, Tolerance,  # noqa: F401
                  SageB200Error, FDR_DTYPE, assign_fdr, device_count, lda_fit)
from .build import build_library, library_path  # noqa: F401
