"""genomics_rs_b200 -- B200-native (sm_100a) affine-gap NW/SW alignment, drop-in for the hot path of
nlaha/genomics-rs (src/alignment/algo.rs).  The product is libgxalign.so (CUDA + C ABI, include/gxalign.h);
this package is the host-side mirror of the reference's interface around it.  No CPU fallback."""
from .config import Config, Scores, get_config, parse_config
from .sequence import Sequence, SequenceContainer
from .alignment import (AlignedSequences, AlignmentChoice, DeviceTable, Plan, RESULT_DTYPE, align, align_all, align_batch,
                        align_reads, alignment_table, k0_measure, pack_pairs, retrace, score_batch, score_planes)
from .banded import Band, band_range, nw_score_banded, nw_score_banded_local
from . import _lib

__all__ = ["Config", "Scores", "get_config", "parse_config", "Sequence", "SequenceContainer", "AlignedSequences",
           "AlignmentChoice", "DeviceTable", "Plan", "RESULT_DTYPE", "align", "align_all", "align_batch", "align_reads",
           "alignment_table", "k0_measure", "pack_pairs", "retrace", "score_batch", "score_planes",
           "Band", "band_range", "nw_score_banded", "nw_score_banded_local"]
