"""ctypes binding of the product library (find_tfbs_b200/libtfbs_b200.so, C ABI in include/tfbs.h).

This is what a host program binds; the Rust driver of the reference would bind the same symbols with
bindgen (INTEGRATION.md).  There is no fallback: if the CUDA library is missing or no B200 is usable,
construction fails loudly.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TFBS_B200_LIB") or os.path.join(_HERE, "libtfbs_b200.so")  # the override is for kernel-variant experiments

TFBS_OK = 0
ERR_INVALID_ARGUMENT, ERR_CUDA, ERR_UNKNOWN_NUCLEOTIDE, ERR_REF_MISMATCH = -1, -2, -3, -4
ERR_MISSING_CASE, ERR_SCORE_RANGE, ERR_STATE, ERR_INTERNAL = -5, -6, -7, -8
ROWS_VARYING, ROWS_ALL_KEYS = 0, 1
PATTERN_PWM, PATTERN_OTHER = 0, 1
DIR_P, DIR_N = 0, 1

EXPORTS = ["tfbs_abi_version", "tfbs_create", "tfbs_destroy", "tfbs_last_error", "tfbs_set_option", "tfbs_set_patterns",
           "tfbs_submit_block", "tfbs_collect", "tfbs_get_matches", "tfbs_upload_block", "tfbs_run_resident", "tfbs_get_stats",
           "tfbs_stream", "tfbs_host_register", "tfbs_host_unregister", "tfbs_audit_block", "tfbs_collect_grouped", "tfbs_expand_rows", "tfbs_set_result_arena",
           "tfbs_merge_sample_blocks", "tfbs_merge_regions", "tfbs_fanout_info", "tfbs_get_attribution"]


class TfbsPattern(C.Structure):
    _fields_ = [("weights", C.POINTER(C.c_int32)), ("len", C.c_uint32), ("min_score", C.c_int32),
                ("pattern_id", C.c_uint16), ("direction", C.c_uint8), ("kind", C.c_uint8)]


class TfbsInnerRegion(C.Structure):
    _fields_ = [("start", C.c_int64), ("end", C.c_int64), ("bed_index", C.c_uint32), ("multiplicity", C.c_uint32)]


class TfbsVariant(C.Structure):
    _fields_ = [("pos", C.c_int64), ("ref_off", C.c_uint32), ("ref_len", C.c_uint32), ("alt_off", C.c_uint32),
                ("alt_len", C.c_uint32), ("carrier_row", C.c_uint32), ("reserved", C.c_uint32)]


class TfbsBlock(C.Structure):
    _fields_ = [("n_regions", C.c_uint32), ("n_samples", C.c_uint32),
                ("region_start", C.POINTER(C.c_int64)), ("region_end", C.POINTER(C.c_int64)),
                ("ref_off", C.POINTER(C.c_uint64)), ("ref_bases", C.POINTER(C.c_uint8)),
                ("inner_off", C.POINTER(C.c_uint32)), ("inner", C.POINTER(TfbsInnerRegion)),
                ("var_off", C.POINTER(C.c_uint32)), ("variants", C.POINTER(TfbsVariant)),
                ("allele_bases", C.POINTER(C.c_uint8)), ("allele_bytes", C.c_uint64),
                ("carriers", C.POINTER(C.c_uint32)), ("n_carrier_rows", C.c_uint32), ("carrier_pitch", C.c_uint32)]


class TfbsRows(C.Structure):
    _fields_ = [("n_rows", C.c_uint64), ("n_samples", C.c_uint32), ("count_bytes", C.c_uint32),
                ("region", C.POINTER(C.c_uint32)), ("inner", C.POINTER(C.c_uint32)), ("pattern_id", C.POINTER(C.c_uint16)),
                ("vmin", C.POINTER(C.c_uint32)), ("vmax", C.POINTER(C.c_uint32)),
                ("left", C.POINTER(C.c_uint32)), ("right", C.POINTER(C.c_uint32))]


class TfbsGroupedRows(C.Structure):
    _fields_ = [("n_rows", C.c_uint64), ("n_samples", C.c_uint32), ("n_regions", C.c_uint32),
                ("region", C.POINTER(C.c_uint32)), ("inner", C.POINTER(C.c_uint32)), ("pattern_id", C.POINTER(C.c_uint16)),
                ("vmin", C.POINTER(C.c_uint32)), ("vmax", C.POINTER(C.c_uint32)), ("base", C.POINTER(C.c_uint32)),
                ("bits", C.POINTER(C.c_uint8)), ("offset", C.POINTER(C.c_uint64)), ("packed", C.POINTER(C.c_uint32)),
                ("packed_words", C.c_uint64), ("n_groups", C.POINTER(C.c_uint32)), ("hap_group", C.c_void_p),
                ("hap_group_bytes", C.c_uint32), ("reserved", C.c_uint32)]


class TfbsArenaHeader(C.Structure):
    _fields_ = [("magic", C.c_uint64), ("sequence", C.c_uint64), ("n_rows", C.c_uint64), ("packed_words", C.c_uint64),
                ("n_samples", C.c_uint32), ("n_regions", C.c_uint32), ("hap_group_bytes", C.c_uint32), ("reserved", C.c_uint32),
                ("off_region", C.c_uint64), ("off_inner", C.c_uint64), ("off_pattern_id", C.c_uint64), ("off_vmin", C.c_uint64),
                ("off_vmax", C.c_uint64), ("off_base", C.c_uint64), ("off_bits", C.c_uint64), ("off_offset", C.c_uint64),
                ("off_packed", C.c_uint64), ("off_n_groups", C.c_uint64), ("off_hap_group", C.c_uint64), ("bytes_used", C.c_uint64)]


ARENA_MAGIC = 0x3152415342465400


def read_arena(buf, half, expand=False):
    """Grouped rows of the block most recently completed in one half of a result arena (tfbs_set_result_arena), e.g. through a
    shared-memory mapping in ANOTHER process than the one that owns the context.  buf: writable/readable uint8 numpy array (or
    np.memmap) over the whole arena."""
    base = (len(buf) // 2) * half
    h = TfbsArenaHeader.from_buffer_copy(bytes(buf[base:base + C.sizeof(TfbsArenaHeader)]))
    if h.magic != ARENA_MAGIC:
        return None
    n, S, R = h.n_rows, h.n_samples, h.n_regions

    def arr(off, cnt, dt):
        return np.frombuffer(buf, dtype=dt, count=cnt, offset=base + off) if cnt else np.zeros(0, dtype=dt)

    hg_dt = np.uint16 if h.hap_group_bytes == 2 else np.uint32
    out = {"sequence": h.sequence, "n_rows": n, "n_samples": S, "n_regions": R, "region": arr(h.off_region, n, np.uint32),
           "inner": arr(h.off_inner, n, np.uint32), "pattern_id": arr(h.off_pattern_id, n, np.uint16), "vmin": arr(h.off_vmin, n, np.uint32),
           "vmax": arr(h.off_vmax, n, np.uint32), "base": arr(h.off_base, n, np.uint32), "bits": arr(h.off_bits, n, np.uint8),
           "offset": arr(h.off_offset, n, np.uint64), "packed": arr(h.off_packed, h.packed_words, np.uint32),
           "n_groups": arr(h.off_n_groups, R, np.uint32), "hap_group": arr(h.off_hap_group, R * 2 * S, hg_dt).reshape(R, 2 * S),
           "bytes": int(h.bytes_used)}
    if expand:
        g = TfbsGroupedRows()
        g.n_rows, g.n_samples, g.n_regions, g.packed_words, g.hap_group_bytes = n, S, R, h.packed_words, h.hap_group_bytes
        keep = []
        for name, ct in (("region", C.c_uint32), ("inner", C.c_uint32), ("pattern_id", C.c_uint16), ("vmin", C.c_uint32), ("vmax", C.c_uint32),
                         ("base", C.c_uint32), ("bits", C.c_uint8), ("offset", C.c_uint64), ("packed", C.c_uint32), ("n_groups", C.c_uint32)):
            a = np.ascontiguousarray(out[name])
            keep.append(a)
            setattr(g, name, a.ctypes.data_as(C.POINTER(ct)))
        hg = np.ascontiguousarray(out["hap_group"])
        g.hap_group = hg.ctypes.data
        left = np.zeros((n, S), dtype=np.uint32)
        right = np.zeros((n, S), dtype=np.uint32)
        if n and lib().tfbs_expand_rows(C.byref(g), 0, n, _ptr(left, C.c_uint32), _ptr(right, C.c_uint32)) != TFBS_OK:
            raise TfbsError(ERR_INVALID_ARGUMENT, "tfbs_expand_rows failed on the arena")
        out["left"], out["right"] = left, right
    return out


_GROUPED_ARRAYS = (("region", C.c_uint32), ("inner", C.c_uint32), ("pattern_id", C.c_uint16), ("vmin", C.c_uint32), ("vmax", C.c_uint32),
                   ("base", C.c_uint32), ("bits", C.c_uint8), ("offset", C.c_uint64), ("packed", C.c_uint32), ("n_groups", C.c_uint32))


def own_grouped(g):
    """Grouped rows (dict of collect_grouped / read_arena) copied into arrays of their own, with a tfbs_grouped_rows over the copies
    under "_c": what a caller keeps when the library's buffers are about to be reused (the next collect)."""
    out = {k: v for k, v in g.items() if k not in ("_c", "_keep")}
    c = TfbsGroupedRows()
    c.n_rows, c.n_samples, c.n_regions = int(g["n_rows"]), int(g["n_samples"]), int(g["n_regions"])
    for name, ct in _GROUPED_ARRAYS:
        a = np.array(g[name], dtype=np.dtype(ct), copy=True)
        out[name] = a
        setattr(c, name, a.ctypes.data_as(C.POINTER(ct)))
    hg = np.array(g["hap_group"], copy=True)
    out["hap_group"] = hg
    c.hap_group = hg.ctypes.data
    c.hap_group_bytes = hg.dtype.itemsize
    c.packed_words = len(out["packed"])
    out["_c"] = c
    return out


def merge_sample_blocks(parts, expand=True):
    """tfbs_merge_sample_blocks over the grouped rows of the sample blocks (dicts with "_c", in sample order): the keys that survive
    min != max over ALL samples; with expand=True the blocks' (left, right) are concatenated along the sample axis
    (tfbs_expand_rows per block and row; a block without the key contributes zeros)."""
    n_parts = len(parts)
    arr = (C.POINTER(TfbsGroupedRows) * max(1, n_parts))(*[C.pointer(p["_c"]) for p in parts])
    n_out = C.c_uint64(0)
    null32, null16, null64 = C.POINTER(C.c_uint32)(), C.POINTER(C.c_uint16)(), C.POINTER(C.c_uint64)()
    rc = lib().tfbs_merge_sample_blocks(arr, n_parts, 0, null32, null32, null16, null32, null32, null64, C.byref(n_out))
    if rc != TFBS_OK:
        raise TfbsError(rc, "tfbs_merge_sample_blocks failed")
    n = n_out.value
    region, inner, pid = np.zeros(n, np.uint32), np.zeros(n, np.uint32), np.zeros(n, np.uint16)
    vmin, vmax, part_row = np.zeros(n, np.uint32), np.zeros(n, np.uint32), np.zeros((max(1, n_parts), n), np.uint64)
    if n:
        rc = lib().tfbs_merge_sample_blocks(arr, n_parts, n, _ptr(region, C.c_uint32), _ptr(inner, C.c_uint32), _ptr(pid, C.c_uint16),
                                            _ptr(vmin, C.c_uint32), _ptr(vmax, C.c_uint32), _ptr(part_row, C.c_uint64), C.byref(n_out))
        if rc != TFBS_OK or n_out.value != n:
            raise TfbsError(rc, "tfbs_merge_sample_blocks failed")
    out = {"region": region, "inner": inner, "pattern_id": pid, "vmin": vmin, "vmax": vmax, "part_row": part_row[:n_parts]}
    if expand:
        lefts, rights = [], []
        for p, part in enumerate(parts):
            S = int(part["n_samples"])
            left, right = np.zeros((n, S), np.uint32), np.zeros((n, S), np.uint32)
            for j in np.nonzero(part_row[p] != np.uint64(0xffffffffffffffff))[0]:
                rc = lib().tfbs_expand_rows(C.byref(part["_c"]), int(part_row[p, j]), 1, _ptr(left[j], C.c_uint32), _ptr(right[j], C.c_uint32))
                if rc != TFBS_OK:
                    raise TfbsError(rc, "tfbs_expand_rows failed")
            lefts.append(left)
            rights.append(right)
        out["left"] = np.concatenate(lefts, axis=1) if lefts else np.zeros((n, 0), np.uint32)
        out["right"] = np.concatenate(rights, axis=1) if rights else np.zeros((n, 0), np.uint32)
    return out


class TfbsMatches(C.Structure):
    _fields_ = [("n_matches", C.c_uint64), ("region", C.POINTER(C.c_uint32)), ("pattern_index", C.POINTER(C.c_uint32)),
                ("group", C.POINTER(C.c_uint32)), ("start", C.POINTER(C.c_int64)), ("hap_group", C.POINTER(C.c_uint32)),
                ("n_samples", C.c_uint32), ("truncated", C.c_uint32)]


class TfbsAudit(C.Structure):
    _fields_ = [("n_ties", C.c_uint64), ("tie_region", C.POINTER(C.c_uint32)), ("tie_pattern_index", C.POINTER(C.c_uint32)),
                ("tie_group", C.POINTER(C.c_uint32)), ("tie_start", C.POINTER(C.c_int64)), ("hap_group", C.POINTER(C.c_uint32)),
                ("hap_flags", C.POINTER(C.c_uint8)), ("n_regions", C.c_uint32), ("n_samples", C.c_uint32),
                ("truncated", C.c_uint32), ("reserved", C.c_uint32)]


HAP_TRUNCATED, HAP_OVERWRITTEN = 1, 2


class TfbsAttribution(C.Structure):
    _fields_ = [("n_rows", C.c_uint64), ("ref_count", C.POINTER(C.c_uint32)), ("term_off", C.POINTER(C.c_uint64)),
                ("term_cfg", C.POINTER(C.c_uint32)), ("term_diff", C.POINTER(C.c_int32)), ("n_cfgs", C.c_uint64),
                ("cfg_region", C.POINTER(C.c_uint32)), ("cfg_flags", C.POINTER(C.c_uint8)), ("cfg_rec_off", C.POINTER(C.c_uint64)),
                ("cfg_rec", C.POINTER(C.c_uint32)), ("n_groups_total", C.c_uint64), ("group_cfg_off", C.POINTER(C.c_uint64)),
                ("group_cfg", C.POINTER(C.c_uint32))]


CFG_TRUNCATES = 1


class TfbsStats(C.Structure):
    _fields_ = [("n_regions", C.c_uint64), ("n_groups", C.c_uint64), ("executed_cells", C.c_uint64), ("nominal_cells", C.c_uint64),
                ("n_hits", C.c_uint64), ("n_keys", C.c_uint64), ("n_rows", C.c_uint64), ("h2d_bytes", C.c_uint64),
                ("d2h_bytes", C.c_uint64), ("scan_launches", C.c_uint32), ("total_launches", C.c_uint32),
                ("ms_group", C.c_float), ("ms_build", C.c_float), ("ms_scan", C.c_float), ("ms_count", C.c_float),
                ("ms_total", C.c_float), ("sm_count", C.c_uint32), ("scan_ctas", C.c_uint32),
                ("evaluated_cells", C.c_uint64), ("n_scan_items", C.c_uint64), ("ms_scan_kernel", C.c_float),
                ("n_dropped", C.c_uint32), ("n_truncated", C.c_uint32), ("reserved", C.c_uint32),
                ("scan_input_bytes", C.c_uint64)]


INNER_DTYPE = np.dtype([("start", "<i8"), ("end", "<i8"), ("bed_index", "<u4"), ("multiplicity", "<u4")])
VARIANT_DTYPE = np.dtype([("pos", "<i8"), ("ref_off", "<u4"), ("ref_len", "<u4"), ("alt_off", "<u4"), ("alt_len", "<u4"),
                          ("carrier_row", "<u4"), ("reserved", "<u4")])


def build(force=False):
    """Compile libtfbs_b200.so for sm_100a with nvcc (in-tree, so that the .so travels with the repo)."""
    csrc = os.path.join(_HERE, "csrc")
    srcs = [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith((".cu", ".cuh", ".cpp", ".hpp")) or f == "Makefile"]
    srcs.append(os.path.join(_HERE, "..", "include", "tfbs.h"))
    if force or not os.path.exists(LIB_PATH) or any(os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in srcs):
        subprocess.check_call(["make", "-C", csrc], stdout=subprocess.DEVNULL)
    return LIB_PATH


_LIB = None


def lib():
    """Load the C-ABI library.  Missing library = hard error (no CPU or PyTorch fallback exists)."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a). "
                               "There is no fallback implementation." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.tfbs_last_error.restype = C.c_char_p
        L.tfbs_last_error.argtypes = [C.c_void_p]
        L.tfbs_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        L.tfbs_destroy.argtypes = [C.c_void_p]
        L.tfbs_destroy.restype = None
        L.tfbs_set_option.argtypes = [C.c_void_p, C.c_char_p, C.c_int64]
        L.tfbs_set_patterns.argtypes = [C.c_void_p, C.POINTER(TfbsPattern), C.c_uint32]
        L.tfbs_submit_block.argtypes = [C.c_void_p, C.POINTER(TfbsBlock)]
        L.tfbs_upload_block.argtypes = [C.c_void_p, C.POINTER(TfbsBlock)]
        L.tfbs_run_resident.argtypes = [C.c_void_p]
        L.tfbs_collect.argtypes = [C.c_void_p, C.POINTER(TfbsRows)]
        L.tfbs_collect_grouped.argtypes = [C.c_void_p, C.POINTER(TfbsGroupedRows)]
        L.tfbs_expand_rows.argtypes = [C.POINTER(TfbsGroupedRows), C.c_uint64, C.c_uint64, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
        L.tfbs_set_result_arena.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        L.tfbs_merge_sample_blocks.argtypes = [C.POINTER(C.POINTER(TfbsGroupedRows)), C.c_uint32, C.c_uint64, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32),
                                               C.POINTER(C.c_uint16), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint64),
                                               C.POINTER(C.c_uint64)]
        L.tfbs_merge_regions.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.c_uint64, C.POINTER(C.c_uint64),
                                         C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        L.tfbs_get_matches.argtypes = [C.c_void_p, C.POINTER(TfbsMatches)]
        L.tfbs_get_stats.argtypes = [C.c_void_p, C.POINTER(TfbsStats)]
        L.tfbs_fanout_info.argtypes = [C.c_void_p] + [C.POINTER(C.c_uint32)] * 4
        L.tfbs_audit_block.argtypes = [C.c_void_p, C.POINTER(TfbsAudit)]
        L.tfbs_get_attribution.argtypes = [C.c_void_p, C.POINTER(TfbsAttribution)]
        L.tfbs_stream.argtypes = [C.c_void_p]
        L.tfbs_stream.restype = C.c_void_p
        L.tfbs_host_register.argtypes = [C.c_void_p, C.c_size_t]
        L.tfbs_host_unregister.argtypes = [C.c_void_p]
        _LIB = L
    return _LIB


class TfbsError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("tfbs error %d: %s" % (code, msg))
        self.code = code
        self.message = msg


def _ptr(a, ctype):
    return a.ctypes.data_as(C.POINTER(ctype))


class PatternSet:
    """pwm_list of the reference (main.rs:237) as a C array; keeps the weight buffers alive."""

    def __init__(self, patterns):
        # patterns: list of dicts {weights: (L,4) int32 | None, min_score, pattern_id, direction, kind}
        self.n = len(patterns)
        self.items = patterns
        self._keep = []
        self.c = (TfbsPattern * max(1, self.n))()
        for i, p in enumerate(patterns):
            kind = p.get("kind", PATTERN_PWM)
            if kind == PATTERN_PWM:
                w = np.ascontiguousarray(np.asarray(p["weights"], dtype=np.int32).reshape(-1, 4))
                self._keep.append(w)
                self.c[i].weights = _ptr(w, C.c_int32)
                self.c[i].len = w.shape[0]
            else:
                self.c[i].weights = None
                self.c[i].len = 0
            self.c[i].min_score = int(p.get("min_score", 0))
            self.c[i].pattern_id = int(p["pattern_id"])
            self.c[i].direction = int(p.get("direction", DIR_P))
            self.c[i].kind = kind


class Block:
    """A tfbs_block over numpy arrays (kept alive by this object)."""

    def __init__(self, n_samples, region_start, region_end, ref_off, ref_bases, inner_off, inner, var_off, variants, allele_bases,
                 carriers):
        self.n_samples = int(n_samples)
        self.region_start = np.ascontiguousarray(region_start, dtype=np.int64)
        self.region_end = np.ascontiguousarray(region_end, dtype=np.int64)
        self.ref_off = np.ascontiguousarray(ref_off, dtype=np.uint64)
        self.ref_bases = np.ascontiguousarray(ref_bases, dtype=np.uint8)
        self.inner_off = np.ascontiguousarray(inner_off, dtype=np.uint32)
        self.inner = np.ascontiguousarray(inner, dtype=INNER_DTYPE)
        self.var_off = np.ascontiguousarray(var_off, dtype=np.uint32)
        self.variants = np.ascontiguousarray(variants, dtype=VARIANT_DTYPE)
        self.allele_bases = np.ascontiguousarray(allele_bases, dtype=np.uint8)
        carriers = np.ascontiguousarray(carriers, dtype=np.uint32)
        if carriers.ndim != 2:
            carriers = carriers.reshape(-1, max(1, (2 * self.n_samples + 31) // 32))
        self.carriers = carriers
        self.n_regions = len(self.region_start)
        b = TfbsBlock()
        b.n_regions = self.n_regions
        b.n_samples = self.n_samples
        b.region_start = _ptr(self.region_start, C.c_int64)
        b.region_end = _ptr(self.region_end, C.c_int64)
        b.ref_off = _ptr(self.ref_off, C.c_uint64)
        b.ref_bases = _ptr(self.ref_bases, C.c_uint8)
        b.inner_off = _ptr(self.inner_off, C.c_uint32)
        b.inner = C.cast(self.inner.ctypes.data, C.POINTER(TfbsInnerRegion))
        b.var_off = _ptr(self.var_off, C.c_uint32)
        b.variants = C.cast(self.variants.ctypes.data, C.POINTER(TfbsVariant))
        b.allele_bases = _ptr(self.allele_bases, C.c_uint8)
        b.allele_bytes = self.allele_bases.size
        b.carriers = _ptr(self.carriers, C.c_uint32)
        b.n_carrier_rows = self.carriers.shape[0]
        b.carrier_pitch = self.carriers.shape[1]
        self.c = b

    def _arrays(self):
        return (self.region_start, self.region_end, self.ref_off, self.ref_bases, self.inner_off, self.inner, self.var_off, self.variants,
                self.allele_bases, self.carriers)

    def pin(self):
        """Page-lock the input arrays (tfbs_host_register) so that H2D copies run at PCIe speed."""
        for a in self._arrays():
            if a.nbytes and lib().tfbs_host_register(a.ctypes.data, a.nbytes) != TFBS_OK:
                raise TfbsError(ERR_CUDA, "cudaHostRegister failed")
        self._pinned = True

    def unpin(self):
        if getattr(self, "_pinned", False):
            for a in self._arrays():
                if a.nbytes:
                    lib().tfbs_host_unregister(a.ctypes.data)
            self._pinned = False

    def input_bytes(self):
        return sum(a.nbytes for a in (self.region_start, self.region_end, self.ref_off, self.ref_bases, self.inner_off, self.inner,
                                      self.var_off, self.variants, self.allele_bases, self.carriers))

    def slice(self, r0, r1, compact=False):
        """Sub-block of regions [r0, r1).  compact=False: variants keep their global carrier rows and allele offsets (the shard
        carries the whole carrier matrix); compact=True: only the carrier rows and allele bytes the shard's records use are kept
        and the records are renumbered -- what a shard sent to another GPU should look like."""
        ro, io, vo = self.ref_off, self.inner_off, self.var_off
        variants = self.variants[int(vo[r0]):int(vo[r1])]
        alleles, carriers = self.allele_bases, self.carriers
        if compact:
            variants = variants.copy()
            if len(variants):
                rows, inv = np.unique(variants["carrier_row"], return_inverse=True)
                carriers = np.ascontiguousarray(self.carriers[rows])
                variants["carrier_row"] = inv.astype(np.uint32)
                lo = int(min(variants["ref_off"].min(), variants["alt_off"].min()))
                hi = int(max((variants["ref_off"] + variants["ref_len"]).max(), (variants["alt_off"] + variants["alt_len"]).max()))
                alleles = np.ascontiguousarray(self.allele_bases[lo:hi])
                variants["ref_off"] -= np.uint32(lo)
                variants["alt_off"] -= np.uint32(lo)
            else:
                carriers = np.zeros((1, self.carriers.shape[1]), dtype=np.uint32)
                alleles = np.zeros(0, dtype=np.uint8)
        return Block(self.n_samples, self.region_start[r0:r1], self.region_end[r0:r1], ro[r0:r1 + 1] - ro[r0],
                     self.ref_bases[int(ro[r0]):int(ro[r1])], io[r0:r1 + 1] - io[r0], self.inner[int(io[r0]):int(io[r1])],
                     vo[r0:r1 + 1] - vo[r0], variants, alleles, carriers)


class Context:
    """tfbs_ctx: one CUDA device, one stream."""

    def __init__(self, device=0):
        self._lib = lib()
        self._h = C.c_void_p()
        rc = self._lib.tfbs_create(device, C.byref(self._h))
        if rc != TFBS_OK:
            raise TfbsError(rc, self._lib.tfbs_last_error(None).decode())
        self._patterns = None

    def close(self):
        if self._h:
            self._lib.tfbs_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != TFBS_OK:
            raise TfbsError(rc, self._lib.tfbs_last_error(self._h).decode())

    def set_option(self, key, value):
        self._check(self._lib.tfbs_set_option(self._h, key.encode(), int(value)))

    def set_patterns(self, pattern_set):
        self._patterns = pattern_set
        self._check(self._lib.tfbs_set_patterns(self._h, pattern_set.c, pattern_set.n))

    def submit_block(self, block):
        self._check(self._lib.tfbs_submit_block(self._h, C.byref(block.c)))

    def upload_block(self, block):
        self._block = block
        self._check(self._lib.tfbs_upload_block(self._h, C.byref(block.c)))

    def run_resident(self):
        self._check(self._lib.tfbs_run_resident(self._h))

    def collect(self, copy=True):
        rows = TfbsRows()
        self._check(self._lib.tfbs_collect(self._h, C.byref(rows)))
        n, S = rows.n_rows, rows.n_samples

        def arr(p, cnt, dt):
            if cnt == 0:
                return np.zeros(0, dtype=dt)
            a = np.ctypeslib.as_array(p, shape=(cnt,))
            return a.astype(dt, copy=True) if copy else a

        ctype, dt = {1: (C.c_uint8, np.uint8), 2: (C.c_uint16, np.uint16), 4: (C.c_uint32, np.uint32)}[rows.count_bytes or 4]

        def counts(p):  # left / right come back as u32 unless option rows_width = 0 chose a narrower type (tfbs_rows.count_bytes)
            if n * S == 0:
                return np.zeros((n, S), dtype=np.uint32)
            a = np.ctypeslib.as_array(C.cast(p, C.POINTER(ctype)), shape=(n * S,)).reshape(n, S)
            return a.astype(np.uint32) if copy else a

        return {"region": arr(rows.region, n, np.uint32), "inner": arr(rows.inner, n, np.uint32),
                "pattern_id": arr(rows.pattern_id, n, np.uint16), "vmin": arr(rows.vmin, n, np.uint32),
                "vmax": arr(rows.vmax, n, np.uint32), "left": counts(rows.left), "right": counts(rows.right),
                "count_bytes": int(rows.count_bytes or 4)}

    def set_result_arena(self, buf):
        """tfbs_set_result_arena: grouped rows are copied by the device straight into `buf` (a uint8 numpy array / np.memmap, e.g.
        over a POSIX shared-memory file that the process gathering the rows has mapped too).  None detaches it."""
        self._arena = buf
        if buf is None:
            self._check(self._lib.tfbs_set_result_arena(self._h, None, 0))
        else:
            self._check(self._lib.tfbs_set_result_arena(self._h, buf.ctypes.data, buf.nbytes))

    def collect_grouped(self, expand=False):
        """tfbs_collect_grouped: the rows with one count per distinct haplotype (group) of the region.  Arrays are views of the
        library's pinned buffers (valid until the next collect); expand=True adds `left` / `right` through tfbs_expand_rows."""
        g = TfbsGroupedRows()
        self._check(self._lib.tfbs_collect_grouped(self._h, C.byref(g)))
        n, S, R = g.n_rows, g.n_samples, g.n_regions

        def arr(p, cnt, ct):
            if cnt == 0:
                return np.zeros(0, dtype=np.dtype(ct))
            return np.ctypeslib.as_array(C.cast(p, C.POINTER(ct)), shape=(cnt,))

        hg_t = C.c_uint16 if g.hap_group_bytes == 2 else C.c_uint32
        out = {"n_rows": n, "n_samples": S, "n_regions": R, "region": arr(g.region, n, C.c_uint32), "inner": arr(g.inner, n, C.c_uint32),
               "pattern_id": arr(g.pattern_id, n, C.c_uint16), "vmin": arr(g.vmin, n, C.c_uint32), "vmax": arr(g.vmax, n, C.c_uint32),
               "base": arr(g.base, n, C.c_uint32), "bits": arr(g.bits, n, C.c_uint8), "offset": arr(g.offset, n, C.c_uint64),
               "packed": arr(g.packed, g.packed_words, C.c_uint32), "n_groups": arr(g.n_groups, R, C.c_uint32),
               "hap_group": arr(g.hap_group, R * 2 * S, hg_t).reshape(R, 2 * S) if R * S else np.zeros((R, 2 * S), np.uint32),
               "bytes": int(n * 31 + g.packed_words * 4 + R * 4 + R * 2 * S * g.hap_group_bytes), "_c": g}
        if expand:
            left = np.zeros((n, S), dtype=np.uint32)
            right = np.zeros((n, S), dtype=np.uint32)
            if n:
                rc = self._lib.tfbs_expand_rows(C.byref(g), 0, n, _ptr(left, C.c_uint32), _ptr(right, C.c_uint32))
                if rc != TFBS_OK:
                    raise TfbsError(rc, "tfbs_expand_rows failed")
            out["left"], out["right"] = left, right
        return out

    def merge_regions(self, ranges):
        """tfbs_merge_regions: the merged regions of the concatenated BED ranges [(start, end)], ascending (bed.rs:37-45)."""
        a = np.ascontiguousarray(np.array(ranges, dtype=np.uint64).reshape(-1, 2))
        n = len(a)
        start, end = np.ascontiguousarray(a[:, 0]), np.ascontiguousarray(a[:, 1])
        o_s, o_e = np.zeros(max(1, n), np.uint64), np.zeros(max(1, n), np.uint64)
        n_out = C.c_uint64(0)
        self._check(self._lib.tfbs_merge_regions(self._h, _ptr(start, C.c_uint64), _ptr(end, C.c_uint64), n, _ptr(o_s, C.c_uint64),
                                                 _ptr(o_e, C.c_uint64), C.byref(n_out)))
        return [(int(o_s[i]), int(o_e[i])) for i in range(n_out.value)]

    def matches(self, n_regions):
        m = TfbsMatches()
        self._check(self._lib.tfbs_get_matches(self._h, C.byref(m)))
        n = m.n_matches

        def arr(p, cnt, dt):
            if cnt == 0:
                return np.zeros(0, dtype=dt)
            return np.ctypeslib.as_array(p, shape=(cnt,)).astype(dt, copy=True)

        return {"region": arr(m.region, n, np.uint32), "pattern_index": arr(m.pattern_index, n, np.uint32),
                "group": arr(m.group, n, np.uint32), "start": arr(m.start, n, np.int64),
                "hap_group": arr(m.hap_group, n_regions * 2 * m.n_samples, np.uint32), "truncated": bool(m.truncated)}

    def audit(self):
        """tfbs_audit_block on the resident block: windows scoring exactly min_score and the per-haplotype flags."""
        a = TfbsAudit()
        self._check(self._lib.tfbs_audit_block(self._h, C.byref(a)))
        n, nh = a.n_ties, a.n_regions * 2 * a.n_samples

        def arr(p, cnt, dt):
            if cnt == 0:
                return np.zeros(0, dtype=dt)
            return np.ctypeslib.as_array(p, shape=(cnt,)).astype(dt, copy=True)

        return {"region": arr(a.tie_region, n, np.uint32), "pattern_index": arr(a.tie_pattern_index, n, np.uint32),
                "group": arr(a.tie_group, n, np.uint32), "start": arr(a.tie_start, n, np.int64),
                "hap_group": arr(a.hap_group, nh, np.uint32), "hap_flags": arr(a.hap_flags, nh, np.uint8),
                "truncated": bool(a.truncated)}

    def attribution(self):
        """tfbs_get_attribution: for the block the last collect returned, per row the reference haplotype's count and the non-zero
        count differences of the configurations (term_off / term_cfg / term_diff), per configuration its region, flags and records
        (indices into the block's variants), per group (block-wide numbering) the configurations its count includes.  NumPy copies."""
        a = TfbsAttribution()
        self._check(self._lib.tfbs_get_attribution(self._h, C.byref(a)))
        n, nc, ng = a.n_rows, a.n_cfgs, a.n_groups_total

        def arr(p, cnt, dt):
            if cnt == 0:
                return np.zeros(0, dtype=dt)
            return np.ctypeslib.as_array(p, shape=(cnt,)).astype(dt, copy=True)

        term_off = arr(a.term_off, n + 1, np.uint64)
        cfg_rec_off = arr(a.cfg_rec_off, nc + 1, np.uint64)
        group_cfg_off = arr(a.group_cfg_off, ng + 1, np.uint64)
        nt, nr, nl = int(term_off[-1]), int(cfg_rec_off[-1]), int(group_cfg_off[-1])
        return {"n_rows": n, "ref_count": arr(a.ref_count, n, np.uint32), "term_off": term_off, "term_cfg": arr(a.term_cfg, nt, np.uint32),
                "term_diff": arr(a.term_diff, nt, np.int32), "n_cfgs": nc, "cfg_region": arr(a.cfg_region, nc, np.uint32),
                "cfg_flags": arr(a.cfg_flags, nc, np.uint8), "cfg_rec_off": cfg_rec_off, "cfg_rec": arr(a.cfg_rec, nr, np.uint32),
                "n_groups_total": ng, "group_cfg_off": group_cfg_off, "group_cfg": arr(a.group_cfg, nl, np.uint32)}

    def stats(self):
        s = TfbsStats()
        self._check(self._lib.tfbs_get_stats(self._h, C.byref(s)))
        return {f: getattr(s, f) for f, _ in TfbsStats._fields_}

    def fanout_info(self):
        """tfbs_fanout_info: the groups a shared-memory count vector holds on this device; for the most recent run, the capacity of
        the count vectors, the CTAs of the fan-out launch and whether the vectors were in device memory."""
        v = [C.c_uint32(0) for _ in range(4)]
        self._check(self._lib.tfbs_fanout_info(self._h, *[C.byref(x) for x in v]))
        return {"smem_groups": v[0].value, "groups_cap": v[1].value, "ctas": v[2].value, "in_device_memory": bool(v[3].value)}

    def stream(self):
        return self._lib.tfbs_stream(self._h)
