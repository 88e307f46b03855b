"""glimmer_mg_b200 -- B200 (sm_100a) implementation of Glimmer-MG's ICM scoring and training hot path.

The product is ``libgmgicm.so`` (hand-written CUDA behind the C-ABI in ``include/gmg_icm.h``).  This
package is the thin Python mirror of the reference's operator surface (``ICM_t`` / ``ICM_Training_t``,
``src/ICM/icm.hh:116-213``) used by the tests and the benchmark; the C++ hosts in ``host/`` link the same
library.  There is no CPU fallback: importing works without a GPU, creating a :class:`Context` does not.
"""
from .icm import (Context, EventModel, ICM, ICMTraining, Params, SeqSet, GmgError, ORF_DTYPE, START_DTYPE, lib, lib_path,
                  build_indep_wo_stops, parse_quality_fasta, regions_from_coords, score_strings_many)

__all__ = ["Context", "EventModel", "ICM", "ICMTraining", "Params", "SeqSet", "GmgError", "ORF_DTYPE", "START_DTYPE", "lib",
           "lib_path", "build_indep_wo_stops", "parse_quality_fasta", "regions_from_coords", "score_strings_many"]
