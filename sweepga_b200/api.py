"""Host-side mirror of the reference's filter interface, over the C ABI.

Names, argument meaning and error behaviour follow the reference:
  FilterConfig                       src/paf_filter.rs:18-49 (live fields)
  PafFilter.new/with_keep_self/with_scaffolds_only/filter_paf/apply_filters
                                     src/paf_filter.rs:239-289, 379-382
  filter_file                        src/unified_filter.rs:280-347
  apply_paf_filter, filter_config_from_align_cfg, parse_filter_mode (library grammar)
                                     src/library_api.rs:31-63, 223-281
  parse_filter_mode_cli, parse_metric_number, parse_identity_value, clamp_scaffold_params, round_nice
                                     src/main.rs:244-293, src/cli.rs:26-130, src/pansn.rs:176-225
  plane_sweep_query/target/both      src/plane_sweep_exact.rs:268-461
Python is only the binding: every compute call goes through libsweepga_b200.so (CUDA, sm_100a).
"""
import ctypes as C
import os
import tempfile
from dataclasses import dataclass, field
from typing import Optional

import numpy as np

from workloads.table import Table, prefix_P, prefix_P2, prefix_ids  # noqa: F401  (pure numpy)

from . import _lib
from ._lib import lib

FilterMode = {"OneToOne": _lib.ONE_TO_ONE, "OneToMany": _lib.ONE_TO_MANY, "ManyToMany": _lib.MANY_TO_MANY}
ScoringFunction = {"Identity": 0, "Length": 1, "LengthIdentity": 2, "LogLengthIdentity": 3, "Matches": 4}
ChainStatus = {0: None, 1: "scaffold", 2: "rescued", 3: "unassigned"}


class SwgError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"sweepga_b200 error {code}: {msg}")
        self.code = code


def _ptr(a, ctype):
    return a.ctypes.data_as(C.POINTER(ctype))


# ------------------------------------------------------------------------------------------------
# flag parsers (host logic in C++, src/host_parsers.cpp)
# ------------------------------------------------------------------------------------------------
def _opt(v):
    return None if v == _lib.NO_LIMIT else int(v)


def parse_filter_mode_cli(s: str):
    """src/main.rs:244-293 -> (mode, max_per_query|None, max_per_target|None); raises on "0" (process::exit)."""
    m, q, t = C.c_uint8(), C.c_uint64(), C.c_uint64()
    rc = lib.swg_parse_filter_mode_cli(s.encode(), C.byref(m), C.byref(q), C.byref(t))
    if rc != 0:
        raise SwgError(rc, f"invalid filter value {s!r}")
    return m.value, _opt(q.value), _opt(t.value)


def parse_filter_mode(s: str):
    """src/library_api.rs:31-63 (the library grammar; differs from the CLI on 'many:1')."""
    m, q, t = C.c_uint8(), C.c_uint64(), C.c_uint64()
    lib.swg_parse_filter_mode_lib(s.encode(), C.byref(m), C.byref(q), C.byref(t))
    return m.value, _opt(q.value), _opt(t.value)


def parse_scoring(s: str) -> int:
    v = C.c_uint8()
    lib.swg_parse_scoring(s.encode(), C.byref(v))
    return v.value


def parse_metric_number(s: str) -> int:
    v = C.c_uint64()
    rc = lib.swg_parse_metric_number(s.encode(), C.byref(v))
    if rc != 0:
        raise ValueError(f"invalid metric number {s!r}")
    return v.value


def parse_identity_value(s: str, ani_percentile: Optional[float] = None) -> float:
    v = C.c_double()
    rc = lib.swg_parse_identity_value(s.encode(), 0 if ani_percentile is None else 1, ani_percentile or 0.0, C.byref(v))
    if rc != 0:
        raise ValueError(f"invalid identity value {s!r}")
    return v.value


ANI_ALL, ANI_ORTHOGONAL, ANI_NPERCENTILE = 0, 1, 2
NSORT_LENGTH, NSORT_IDENTITY, NSORT_SCORE = 0, 1, 2


def parse_ani_method(s: str):
    """parse_ani_method (src/main.rs:296-331) -> (method, percentile, sort) or None."""
    m, p, k = C.c_int(), C.c_double(), C.c_int()
    if lib.swg_parse_ani_method(s.encode(), C.byref(m), C.byref(p), C.byref(k)) != 0:
        return None
    return m.value, p.value, k.value


def ani_stats(ctx: "Context", paf_path: str, method="n100"):
    """calculate_ani_stats (src/main.rs:334-688) on the GPU -> (ani50, n_genome_pairs).  `method` is the --ani-method string
    ("all", "orthogonal", "n50", "n90-length", ...; unknown strings fall back to n50-identity like the CLI) or a tuple."""
    if isinstance(method, str):
        method = parse_ani_method(method) or (ANI_NPERCENTILE, 50.0, NSORT_IDENTITY)
    ani, npairs = C.c_double(), C.c_uint64()
    ctx._check(lib.swg_ani_stats(ctx._h, os.fsencode(paf_path), int(method[0]), float(method[1]), int(method[2]), C.byref(ani), C.byref(npairs)))
    return ani.value, int(npairs.value)


def apply_tree_filter_to_paf(ctx: "Context", input_path: str, output_path: str, k_nearest: int, k_farthest: int = 0,
                             random_fraction: float = 0.0):
    """apply_tree_filter_to_paf (src/tree_filter.rs:205-283) on the GPU -> (lines kept, genome pairs selected)."""
    kept, sel = C.c_uint64(), C.c_uint64()
    ctx._check(lib.swg_tree_filter_paf(ctx._h, os.fsencode(input_path), os.fsencode(output_path), int(k_nearest), int(k_farthest),
                                       float(random_fraction), C.byref(kept), C.byref(sel)))
    return int(kept.value), int(sel.value)


def round_nice(v: int) -> int:
    return lib.swg_round_nice(v)


def clamp_scaffold_params(user_jump, user_mass, avg_seq_len, adaptive):
    j, m = C.c_uint64(), C.c_uint64()
    lib.swg_clamp_scaffold_params(user_jump, user_mass, 0 if avg_seq_len is None else 1, avg_seq_len or 0, 1 if adaptive else 0,
                                  C.byref(j), C.byref(m))
    return j.value, m.value


# ------------------------------------------------------------------------------------------------
@dataclass
class FilterConfig:
    """Live fields of the reference FilterConfig (src/paf_filter.rs:18-49); defaults = CLI defaults."""
    min_block_length: int = 0
    mapping_filter_mode: int = _lib.MANY_TO_MANY
    mapping_max_per_query: Optional[int] = None
    mapping_max_per_target: Optional[int] = None
    scaffold_filter_mode: int = _lib.MANY_TO_MANY
    scaffold_max_per_query: Optional[int] = None
    scaffold_max_per_target: Optional[int] = None
    overlap_threshold: float = 0.95
    scaffold_gap: int = 50_000
    min_scaffold_length: int = 10_000
    scaffold_overlap_threshold: float = 0.5
    scaffold_max_deviation: int = 0
    scoring_function: int = _lib.SCORE_LOG_LENGTH_IDENTITY
    min_identity: float = 0.0
    min_scaffold_identity: float = 0.0
    keep_self: bool = False        # PafFilter::with_keep_self
    scaffolds_only: bool = False   # PafFilter::with_scaffolds_only

    @classmethod
    def from_cli(cls, num_mappings="many:many", scaffold_filter="many:many", scoring="log-length-ani", overlap=0.95,
                 scaffold_overlap=0.5, scaffold_jump="50k", scaffold_mass="10k", scaffold_dist="0", min_aln_length=None,
                 min_aln_identity="0", min_scaffold_identity="0", keep_self=False, scaffolds_only=False,
                 avg_seq_len=None, no_adaptive_scaffolds=False, ani_percentile=None):
        """The CLI's FilterConfig construction (src/main.rs:3476-3619), flag strings in, config out."""
        mm, mq, mt = parse_filter_mode_cli(str(num_mappings))
        sm, sq, st = parse_filter_mode_cli(str(scaffold_filter))
        jump = parse_metric_number(str(scaffold_jump))
        mass = parse_metric_number(str(scaffold_mass))
        jump, mass = clamp_scaffold_params(jump, mass, avg_seq_len, not no_adaptive_scaffolds)
        mid = parse_identity_value(str(min_aln_identity), ani_percentile)
        msid = mid if str(min_scaffold_identity) == "" else parse_identity_value(str(min_scaffold_identity), ani_percentile)
        return cls(min_block_length=0 if min_aln_length is None else parse_metric_number(str(min_aln_length)),
                   mapping_filter_mode=mm, mapping_max_per_query=mq, mapping_max_per_target=mt,
                   scaffold_filter_mode=sm, scaffold_max_per_query=sq, scaffold_max_per_target=st,
                   overlap_threshold=float(overlap), scaffold_gap=jump, min_scaffold_length=mass,
                   scaffold_overlap_threshold=float(scaffold_overlap), scaffold_max_deviation=parse_metric_number(str(scaffold_dist)),
                   scoring_function=parse_scoring(scoring), min_identity=mid, min_scaffold_identity=msid,
                   keep_self=keep_self, scaffolds_only=scaffolds_only)

    def to_c(self) -> _lib.swg_config:
        c = _lib.swg_config()
        n = lambda v: _lib.NO_LIMIT if v is None else int(v)
        c.min_block_length = int(self.min_block_length)
        c.mapping_max_per_query, c.mapping_max_per_target = n(self.mapping_max_per_query), n(self.mapping_max_per_target)
        c.scaffold_max_per_query, c.scaffold_max_per_target = n(self.scaffold_max_per_query), n(self.scaffold_max_per_target)
        c.scaffold_gap, c.min_scaffold_length = int(self.scaffold_gap), int(self.min_scaffold_length)
        c.scaffold_max_deviation = int(self.scaffold_max_deviation)
        c.overlap_threshold, c.scaffold_overlap_threshold = float(self.overlap_threshold), float(self.scaffold_overlap_threshold)
        c.min_identity, c.min_scaffold_identity = float(self.min_identity), float(self.min_scaffold_identity)
        c.mapping_filter_mode, c.scaffold_filter_mode = int(self.mapping_filter_mode), int(self.scaffold_filter_mode)
        c.scoring_function = int(self.scoring_function)
        c.keep_self, c.scaffolds_only = int(bool(self.keep_self)), int(bool(self.scaffolds_only))
        return c


def filter_config_from_align_cfg(num_mappings="many:many", scaffold_filter="many:many", scaffold_jump=50_000,
                                 scaffold_mass=10_000, scaffold_dist=0, overlap=0.95, min_identity=0.0, min_map_length=0,
                                 avg_seq_len=0) -> FilterConfig:
    """src/library_api.rs:223-259: library grammar, adaptive clamp always on, scaffold overlap fixed at 0.5,
    LogLengthIdentity, min_scaffold_identity = min_identity."""
    mm, mq, mt = parse_filter_mode(num_mappings)
    sm, sq, st = parse_filter_mode(scaffold_filter)
    jump, mass = clamp_scaffold_params(scaffold_jump, scaffold_mass, avg_seq_len if avg_seq_len > 0 else None, True)
    return FilterConfig(min_block_length=min_map_length, mapping_filter_mode=mm, mapping_max_per_query=mq, mapping_max_per_target=mt,
                        scaffold_filter_mode=sm, scaffold_max_per_query=sq, scaffold_max_per_target=st, overlap_threshold=overlap,
                        scaffold_gap=jump, min_scaffold_length=mass, scaffold_overlap_threshold=0.5,
                        scaffold_max_deviation=scaffold_dist, scoring_function=_lib.SCORE_LOG_LENGTH_IDENTITY,
                        min_identity=min_identity, min_scaffold_identity=min_identity)


# ------------------------------------------------------------------------------------------------
class MappingTable(Table):
    """The compact SoA that replaces Vec<RecordMeta> (include/sweepga_b200.h: swg_mappings): the numpy column table of
    `workloads.table.Table` plus its ctypes view.  `identity=None` leaves swg_mappings.identity NULL: the device then
    derives matches / max(block_length, 1) itself (src/paf_filter.rs:322)."""

    def to_c(self) -> _lib.swg_mappings:
        m = _lib.swg_mappings()
        m.n = self.n
        for f in ("query_id", "target_id", "query_start", "query_end", "target_start", "target_end", "block_length", "matches",
                  "seq_genome_id", "seq_genome2_id"):
            setattr(m, f, _ptr(getattr(self, f), C.c_uint32))
        if getattr(self, "ids16", None) is not None:  # (query_id16, target_id16): 2 B per id on the wire (n_seq <= 65536)
            m.query_id, m.target_id = None, None
            m.query_id16, m.target_id16 = _ptr(self.ids16[0], C.c_uint16), _ptr(self.ids16[1], C.c_uint16)
        m.identity = _ptr(self.identity, C.c_double) if self.identity is not None else None
        m.strand = _ptr(self.strand, C.c_uint8)
        m.score = _ptr(self.score, C.c_double) if self.score is not None else None
        m.n_seq = self.n_seq
        return m


# ------------------------------------------------------------------------------------------------
def with_ids16(table: "MappingTable", alloc=None) -> "MappingTable":
    """A copy of the table whose swg_mappings view carries 16-bit id columns (n_seq <= 65536).  alloc(array) -> array lets the
    caller place the two columns (e.g. in pinned memory)."""
    import copy
    if table.n_seq > 65536:
        raise ValueError(f"16-bit id columns hold at most 65536 sequences, the table has {table.n_seq}")
    t = copy.copy(table)
    q, tt = table.query_id.astype(np.uint16), table.target_id.astype(np.uint16)
    t.ids16 = (alloc(q), alloc(tt)) if alloc else (q, tt)
    return t


class Context:
    """swg_ctx: one per GPU.  Raises (never falls back) when no sm_100 device is usable."""

    def __init__(self, device: int = 0):
        self._h = lib.swg_create(device)
        if not self._h:
            raise SwgError(_lib.ERR_CUDA, (lib.swg_last_error(None) or b"").decode())

    def close(self):
        if self._h:
            lib.swg_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise SwgError(rc, (lib.swg_last_error(self._h) or b"").decode())

    def filter(self, cfg: FilterConfig, table: MappingTable, status=None, chain_id=None):
        """apply_filters on HOST buffers (H2D + kernels + D2H).  Returns (status u8[n], chain_id u32[n], stats)."""
        n = table.n
        status = np.zeros(n, np.uint8) if status is None else status
        chain_id = np.zeros(n, np.uint32) if chain_id is None else chain_id
        res = _lib.swg_result(_ptr(status, C.c_uint8), _ptr(chain_id, C.c_uint32))
        stats = _lib.swg_stats()
        cm, cc = table.to_c(), cfg.to_c()
        self._check(lib.swg_filter(self._h, C.byref(cc), C.byref(cm), C.byref(res), C.byref(stats)))
        return status, chain_id, stats

    def filter_batch(self, cfg: FilterConfig, tables):
        """Many independent tables in one call (swg_filter_batch): every table's result is what filter() returns for it alone.
        Returns (results, counts, stats): results[k] = (status u8[n_k], chain_id u32[n_k]); counts = uint64 (K, TC_COUNT), columns
        TC_STAGE1, TC_KEPT, TC_SCAFFOLD, TC_RESCUED, TC_CHAINS_KEPT; stats describes the whole call."""
        tables = list(tables)
        k = len(tables)
        results = [(np.zeros(t.n, np.uint8), np.zeros(t.n, np.uint32)) for t in tables]
        cms = (_lib.swg_mappings * max(k, 1))(*[t.to_c() for t in tables])
        outs = (_lib.swg_result * max(k, 1))(*[_lib.swg_result(_ptr(s, C.c_uint8), _ptr(c, C.c_uint32)) for s, c in results])
        counts = np.zeros((k, _lib.TC_COUNT), np.uint64)
        stats = _lib.swg_stats()
        cc = cfg.to_c()
        self._check(lib.swg_filter_batch(self._h, C.byref(cc), k, cms, outs, _ptr(counts, C.c_uint64), C.byref(stats)))
        return results, counts, stats

    def filter_paf_batch(self, cfg: FilterConfig, in_paths, out_paths):
        """Many independent PAF files in one call (swg_filter_paf_batch): out_paths[k] receives what swg_filter_paf writes for
        in_paths[k] alone.  Returns (counts, stats): counts = uint64 (K, TC_COUNT) as in filter_batch; stats describes the call."""
        ins = [os.fsencode(p) for p in in_paths]
        outs = [os.fsencode(p) for p in out_paths]
        if len(ins) != len(outs):
            raise ValueError("filter_paf_batch: in_paths and out_paths differ in length")
        k = len(ins)
        cin = (C.c_char_p * max(k, 1))(*ins)
        cout = (C.c_char_p * max(k, 1))(*outs)
        counts = np.zeros((k, _lib.TC_COUNT), np.uint64)
        stats = _lib.swg_stats()
        cc = cfg.to_c()
        self._check(lib.swg_filter_paf_batch(self._h, C.byref(cc), k, cin, cout, _ptr(counts, C.c_uint64), C.byref(stats)))
        return counts, stats

    def prefetch(self, table: MappingTable):
        """Start uploading `table` now (swg_prefetch); the next filter() of the same table (same arrays) finds it on the device."""
        cm = table.to_c()
        self._check(lib.swg_prefetch(self._h, C.byref(cm)))

    def prefetch_drop(self):
        lib.swg_prefetch_drop(self._h)

    def upload(self, table: MappingTable):
        dev, dres = _lib.swg_mappings(), _lib.swg_result()
        cm = table.to_c()
        self._check(lib.swg_upload(self._h, C.byref(cm), C.byref(dev), C.byref(dres)))
        return dev, dres

    def filter_device(self, cfg: FilterConfig, dev, dres):
        stats = _lib.swg_stats()
        cc = cfg.to_c()
        self._check(lib.swg_filter_device(self._h, C.byref(cc), C.byref(dev), C.byref(dres), C.byref(stats)))
        return stats

    def download(self, n, dres):
        status, chain_id = np.zeros(n, np.uint8), np.zeros(n, np.uint32)
        res = _lib.swg_result(_ptr(status, C.c_uint8), _ptr(chain_id, C.c_uint32))
        self._check(lib.swg_download_result(self._h, n, C.byref(dres), C.byref(res)))
        return status, chain_id

    def score_column(self, identity, query_start, query_end, scoring=3):
        """score_with_function (src/plane_sweep_exact.rs:29-86) of every row, evaluated on the device (swg_score_column)."""
        idy = np.ascontiguousarray(identity, np.float64)
        qs, qe = np.ascontiguousarray(query_start, np.uint32), np.ascontiguousarray(query_end, np.uint32)
        out = np.empty(len(idy), np.float64)
        self._check(lib.swg_score_column(self._h, len(idy), _ptr(idy, C.c_double), _ptr(qs, C.c_uint32), _ptr(qe, C.c_uint32), int(scoring),
                                         _ptr(out, C.c_double)))
        return out

    def chain_identity(self, total_length, sum_block, sum_matches):
        """weighted_identity of chains (src/paf_filter.rs:896-913), evaluated on the device (swg_chain_identity)."""
        a = [np.ascontiguousarray(x, np.uint64) for x in (total_length, sum_block, sum_matches)]
        out = np.empty(len(a[0]), np.float64)
        self._check(lib.swg_chain_identity(self._h, len(a[0]), *[_ptr(x, C.c_uint64) for x in a], _ptr(out, C.c_double)))
        return out

    def log_matches_host(self) -> bool:
        """True when the device's ln() produced the host libm's bits on the probe set of swg_create."""
        return lib.swg_log_matches_host(self._h) == 1

    def last_chain_keys(self):
        """Order keys (A, B) of the chains kept by the last filter call on this context (swg_last_chain_keys)."""
        n = C.c_uint64()
        lib.swg_last_chain_keys(self._h, 0, None, None, C.byref(n))  # cap 0: only the count is reported
        k = int(n.value)
        if k == 0:
            return np.zeros(0, np.uint32), np.zeros(0, np.uint32)
        a, b = np.zeros(k, np.uint32), np.zeros(k, np.uint32)
        self._check(lib.swg_last_chain_keys(self._h, k, _ptr(a, C.c_uint32), _ptr(b, C.c_uint32), C.byref(n)))
        return a, b

    def last_chain_units(self, max_units=0):
        """Runs of kept chains that share a genome-pair unit, for the last call (swg_last_chain_units):
        (A = input index of the unit's first stage-1 record, first local chain number of the run), in chain order.
        max_units: an upper bound on the number of runs if the caller knows one (one round trip instead of two)."""
        n = C.c_uint64()
        if not max_units:
            self._check(lib.swg_last_chain_units(self._h, 0, None, None, C.byref(n)))
            max_units = int(n.value)
        a, f = np.zeros(max(max_units, 1), np.uint32), np.zeros(max(max_units, 1), np.uint32)
        if max_units:
            self._check(lib.swg_last_chain_units(self._h, max_units, _ptr(a, C.c_uint32), _ptr(f, C.c_uint32), C.byref(n)))
        k = int(n.value)
        return a[:k], f[:k]

    def renumber_chains_device(self, n, chain_id_dev_ptr, unit_first_chain, unit_delta):
        fk = np.ascontiguousarray(unit_first_chain, np.uint32)
        dl = np.ascontiguousarray(unit_delta, np.int64)
        self._check(lib.swg_renumber_chains_device(self._h, n, chain_id_dev_ptr, len(fk), _ptr(fk, C.c_uint32), _ptr(dl, C.c_int64)))

    def pack_status_device(self, n, status_dev_ptr, packed_dev_ptr):
        self._check(lib.swg_pack_status_device(self._h, n, status_dev_ptr, packed_dev_ptr))

    def release(self, dev, dres):
        lib.swg_release(self._h, C.byref(dev), C.byref(dres))

    def stream(self):
        return lib.swg_stream(self._h)

    # plane_sweep_exact.rs:268-461 -> list of kept local indices (ascending), like the reference's Vec<usize>
    def _sweep(self, fn, mappings, *tail):
        qs, qe, ts, te, idy = (np.ascontiguousarray([m[k] for m in mappings], dtype=dt)
                               for k, dt in ((0, np.uint32), (1, np.uint32), (2, np.uint32), (3, np.uint32), (4, np.float64)))
        keep = np.zeros(len(mappings), np.uint8)
        self._check(fn(self._h, len(mappings), _ptr(qs, C.c_uint32), _ptr(qe, C.c_uint32), _ptr(ts, C.c_uint32), _ptr(te, C.c_uint32),
                       _ptr(idy, C.c_double), *tail, _ptr(keep, C.c_uint8)))
        return [int(i) for i in np.nonzero(keep)[0]]

    def plane_sweep_query(self, mappings, mappings_to_keep, overlap_threshold, scoring=3):
        return self._sweep(lib.swg_plane_sweep_query, mappings, _n(mappings_to_keep), overlap_threshold, scoring)

    def plane_sweep_target(self, mappings, mappings_to_keep, overlap_threshold, scoring=3):
        return self._sweep(lib.swg_plane_sweep_target, mappings, _n(mappings_to_keep), overlap_threshold, scoring)

    def plane_sweep_both(self, mappings, query_to_keep, target_to_keep, overlap_threshold, scoring=3):
        return self._sweep(lib.swg_plane_sweep_both, mappings, _n(query_to_keep), _n(target_to_keep), overlap_threshold, scoring)


    def plane_sweep_core(self, intervals, max_to_keep, overlap_threshold):
        """plane_sweep_core::plane_sweep on [(begin, end, score), ...] -> kept indices in the reference's order."""
        n = len(intervals)
        b = np.ascontiguousarray([i[0] for i in intervals], dtype=np.uint32)
        e = np.ascontiguousarray([i[1] for i in intervals], dtype=np.uint32)
        s = np.ascontiguousarray([i[2] for i in intervals], dtype=np.float64)
        out = np.zeros(max(n, 1), np.uint64)
        cnt = C.c_uint64()
        self._check(lib.swg_plane_sweep_core(self._h, n, _ptr(b, C.c_uint32), _ptr(e, C.c_uint32), _ptr(s, C.c_double), _n(max_to_keep),
                                             overlap_threshold, _ptr(out, C.c_uint64), C.byref(cnt)))
        return [int(x) for x in out[: cnt.value]]


class MultiContext:
    """swg_multi: one context per listed GPU behind one call; results identical to a single-GPU call (chain numbers too)."""

    def __init__(self, devices):
        arr = (C.c_int * len(devices))(*devices)
        self._h = lib.swg_multi_create(arr, len(devices))
        if not self._h:
            raise SwgError(_lib.ERR_CUDA, (lib.swg_last_error(None) or b"").decode())

    def close(self):
        if self._h:
            lib.swg_multi_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def filter(self, cfg: FilterConfig, table: MappingTable):
        n = table.n
        status, chain_id = np.zeros(n, np.uint8), np.zeros(n, np.uint32)
        res = _lib.swg_result(_ptr(status, C.c_uint8), _ptr(chain_id, C.c_uint32))
        stats = _lib.swg_stats()
        cm, cc = table.to_c(), cfg.to_c()
        rc = lib.swg_multi_filter(self._h, C.byref(cc), C.byref(cm), C.byref(res), C.byref(stats))
        if rc != 0:
            raise SwgError(rc, (lib.swg_multi_last_error(self._h) or b"").decode())
        return status, chain_id, stats


USIZE_MAX = (1 << 64) - 1


def _n(v):
    return USIZE_MAX if v is None else int(v)


# ------------------------------------------------------------------------------------------------
def parse_paf(path: str, ctx: "Context" = None) -> MappingTable:
    """extract_metadata (src/paf_filter.rs:292-376) -> MappingTable (+ rank, names).  With a Context the text is
    tokenised on the GPU (swg_paf_parse_device), without one on all host threads (swg_paf_parse)."""
    if ctx is not None:
        h = lib.swg_paf_parse_device(ctx._h, os.fsencode(path))
        if not h:
            raise SwgError(_lib.ERR_IO, lib.swg_last_error(ctx._h).decode())
    else:
        err = C.create_string_buffer(256)
        h = lib.swg_paf_parse(os.fsencode(path), err, 256)
        if not h:
            raise SwgError(_lib.ERR_IO, err.value.decode())
    try:
        m = _lib.swg_mappings()
        lib.swg_paf_view(h, C.byref(m))
        n, ns = int(m.n), int(m.n_seq)
        cp = lambda p, cnt, dt: np.ctypeslib.as_array(p, shape=(cnt,)).astype(dt, copy=True) if cnt else np.zeros(0, dt)
        t = MappingTable(cp(m.query_id, n, np.uint32), cp(m.target_id, n, np.uint32), cp(m.query_start, n, np.uint32),
                         cp(m.query_end, n, np.uint32), cp(m.target_start, n, np.uint32), cp(m.target_end, n, np.uint32),
                         cp(m.block_length, n, np.uint32), cp(m.matches, n, np.uint32), cp(m.identity, n, np.float64),
                         cp(m.strand, n, np.uint8), cp(m.seq_genome_id, ns, np.uint32), cp(m.seq_genome2_id, ns, np.uint32))
        t.names = [lib.swg_paf_seq_name(h, i).decode() for i in range(ns)]
        t.rank = cp(lib.swg_paf_rank(h), n, np.uint64)
        return t
    finally:
        lib.swg_paf_free(h)


class PafFilter:
    """PafFilter (src/paf_filter.rs:229-289).  `device` picks the GPU; there is no CPU path."""

    def __init__(self, config: FilterConfig, device: int = 0):
        self.config = FilterConfig(**vars(config))  # keep_self / scaffolds_only ride along (builder methods below override)
        self.device = device
        self._ctx = None

    @classmethod
    def new(cls, config: FilterConfig, device: int = 0):
        return cls(config, device)

    def with_keep_self(self, keep_self: bool):
        self.config.keep_self = bool(keep_self)
        return self

    def with_scaffolds_only(self, scaffolds_only: bool):
        self.config.scaffolds_only = bool(scaffolds_only)
        return self

    def _context(self):
        if self._ctx is None:
            self._ctx = Context(self.device)
        return self._ctx

    def filter_paf(self, input_path: str, output_path: str, host_frontend: bool = False):
        """filter_paf (src/paf_filter.rs:278-289).  The text is tokenised and the tagged output assembled on the GPU;
        host_frontend=True runs the multi-threaded host parser / writer around the same filter instead."""
        ctx = self._context()
        stats = _lib.swg_stats()
        cc = self.config.to_c()
        fn = lib.swg_filter_paf_host if host_frontend else lib.swg_filter_paf
        ctx._check(fn(ctx._h, C.byref(cc), os.fsencode(input_path), os.fsencode(output_path), C.byref(stats)))
        return stats

    def apply_filters(self, table: MappingTable):
        """-> {index: (chain_id or None, status)} like HashMap<rank, RecordMeta>; index = position in `table`
        (or the PAF rank when the table came from parse_paf)."""
        status, chain, _ = self._context().filter(self.config, table)
        keys = table.rank if table.rank is not None else np.arange(table.n)
        return {int(keys[i]): (f"chain_{int(chain[i])}" if chain[i] else None, ChainStatus[int(status[i])])
                for i in np.nonzero(status)[0]}


def filter_file(input_path, output_path, config: FilterConfig, force_paf_output=False, keep_self=False, device=0):
    """unified_filter::filter_file (src/unified_filter.rs:280-347).  A .1aln input is converted through FastGA's ALNtoPAF when
    that executable is found ($SWG_ALNTOPAF or PATH) and the output path ends in ".paf" (src/main.rs:737-770); otherwise, and for
    .1aln output, SwgError(UNSUPPORTED)."""
    with Context(device) as ctx:
        stats = _lib.swg_stats()
        cc = config.to_c()
        ctx._check(lib.swg_filter_file(ctx._h, C.byref(cc), os.fsencode(input_path), os.fsencode(output_path), int(keep_self),
                                       C.byref(stats)))
        return stats


def aln_to_paf(aln_path, paf_path, threads=8):
    """aln_to_paf's fallback (src/main.rs:743-770): `ALNtoPAF -x -T<threads> <aln>` -> paf_path.  Host only."""
    rc = lib.swg_aln_to_paf(os.fsencode(aln_path), os.fsencode(paf_path), int(threads))
    if rc != 0:
        raise SwgError(rc, "no ALNtoPAF executable ($SWG_ALNTOPAF / PATH)" if rc == _lib.ERR_UNSUPPORTED else "ALNtoPAF failed")


def apply_paf_filter(paf_path: str, filter_config: FilterConfig, device=0) -> str:
    """library_api::apply_paf_filter (src/library_api.rs:267-281): returns the path of a new filtered temp file."""
    fd, out = tempfile.mkstemp(suffix=".filtered.paf")
    os.close(fd)
    PafFilter(filter_config, device).with_keep_self(False).filter_paf(paf_path, out)
    return out


def shard_plan_units(unit_sizes, n_shards: int):
    """swg_shard_plan_units: LPT of unit sizes -> (shard_of_unit, shard_sizes)."""
    us = np.ascontiguousarray(unit_sizes, np.uint64)
    so = np.zeros(len(us), np.uint32)
    sizes = np.zeros(n_shards, np.uint64)
    rc = lib.swg_shard_plan_units(len(us), _ptr(us, C.c_uint64), n_shards, _ptr(so, C.c_uint32), _ptr(sizes, C.c_uint64))
    if rc != 0:
        raise SwgError(rc, "swg_shard_plan_units")
    return so, sizes


def shard_plan(table: MappingTable, n_shards: int):
    """Size-balanced genome-pair sharding for the multi-GPU driver -> (shard_of[n], shard_sizes[n_shards])."""
    shard_of = np.zeros(table.n, np.uint32)
    sizes = np.zeros(n_shards, np.uint64)
    cm = table.to_c()
    rc = lib.swg_shard_plan(C.byref(cm), n_shards, _ptr(shard_of, C.c_uint32), _ptr(sizes, C.c_uint64))
    if rc != 0:
        raise SwgError(rc, "swg_shard_plan")
    return shard_of, sizes
