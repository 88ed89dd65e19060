"""sweepga_b200 — B200-native (sm_100a) implementation of sweepga's mapping-filter hot path.

The product is libsweepga_b200.so (C ABI in include/sweepga_b200.h, CUDA kernels in csrc/); this package
is the host-side mirror of the reference's filter interface over that ABI.  No CPU fallback exists.
"""
from . import _lib
from ._lib import lib, DROPPED, SCAFFOLD, RESCUED, UNASSIGNED, TC_STAGE1, TC_KEPT, TC_SCAFFOLD, TC_RESCUED, TC_CHAINS_KEPT, TC_COUNT
from .api import (ChainStatus, Context, MultiContext, FilterConfig, FilterMode, MappingTable, PafFilter, ScoringFunction, SwgError,
                  apply_paf_filter, clamp_scaffold_params, filter_config_from_align_cfg, filter_file, parse_filter_mode,
                  parse_filter_mode_cli, parse_identity_value, parse_metric_number, parse_paf, parse_scoring, prefix_P,
                  prefix_P2, prefix_ids, round_nice, shard_plan, shard_plan_units, with_ids16, ani_stats, parse_ani_method, ANI_ALL, ANI_ORTHOGONAL,
                  ANI_NPERCENTILE, NSORT_LENGTH, NSORT_IDENTITY, NSORT_SCORE, apply_tree_filter_to_paf)

__version__ = lib.swg_version().decode()
