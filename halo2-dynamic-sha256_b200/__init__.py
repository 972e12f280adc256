"""halo2-dynamic-sha256_b200 -- host-side mirror of the reference's chip API over the C-ABI engine.

The reference (zhmolly/halo2-dynamic-sha256) is a Rust crate; no Rust toolchain exists in this image, so the
host side above the C-ABI (include/h2sha_b200.h, built from csrc/) is mirrored here in Python for the tests
and the benchmark, and in C++ (csrc/host_api.hpp) / Rust source (rust/) for integrators.  Names, argument
meaning and error behaviour follow `Sha256DynamicConfig` (reference src/lib.rs:38-369):

    configure(max_variable_byte_sizes, range..., num_bits_lookup, num_advice_columns, is_input_range_check)   lib.rs:49-56
    digest(input, precomputed_input_len) -> AssignedHashResult{input_len, input_bytes, output_bytes}          lib.rs:71-76

PyTorch is used only to own device memory and streams; all compute happens in libh2sha_b200.so.  There is no
CPU fallback: without a GPU only the static plan (layout, shape, handles) can be queried (`device=-1`); every
witness-generating call raises `EngineError`.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libh2sha_b200.so")

H2SHA_OK, H2SHA_EINVAL, H2SHA_EPANIC, H2SHA_ECUDA, H2SHA_ENOMEM = 0, -1, -2, -3, -4

# symbols include/h2sha_b200.h declares (checked by tests/test_abi.py)
EXPORTED_SYMBOLS = [
    "h2sha_create", "h2sha_destroy", "h2sha_last_error", "h2sha_build_id", "h2sha_get_layout", "h2sha_get_breaks", "h2sha_get_handles", "h2sha_get_digest_ranges", "h2sha_get_shape", "h2sha_get_lookup_tables",
    "h2sha_digest_batch", "h2sha_export_instance", "h2sha_export_batch", "h2sha_get_compact_info", "h2sha_get_compact_map", "h2sha_expand_compact", "h2sha_get_lookup_info", "h2sha_lookup_multiplicities", "h2sha_permute_lookup", "h2sha_permute_lookup_from_raw", "h2sha_lookup_product", "h2sha_get_permutation", "h2sha_permutation_product", "h2sha_permute_lookup_per_instance", "h2sha_permute_lookup_from_raw_per_instance", "h2sha_lookup_product_per_instance", "h2sha_permutation_product_per_instance", "h2sha_check_batch", "h2sha_check_batch_per_instance", "h2sha_check_site", "h2sha_gather", "h2sha_zero_outputs", "h2sha_debug_mont_from_u64", "h2sha_debug_mont_from_u32", "h2sha_debug_store_probe", "h2sha_debug_int_probe", "h2sha_last_launch_count", "h2sha_last_kernel_ms", "H2SHA_CK_M",
]


class EngineError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"h2sha error {code}: {msg}")
        self.code = code


class ReferencePanic(EngineError):
    """Input on which the reference panics (lib.rs:89-90)."""


class _Config(C.Structure):
    _fields_ = [("n_digests", C.c_uint32), ("max_variable_byte_sizes", C.POINTER(C.c_uint32)), ("max_rows", C.c_uint32),
                ("lookup_bits", C.c_uint32), ("num_bits_lookup", C.c_uint32), ("num_advice_columns", C.c_uint32),
                ("is_input_range_check", C.c_uint32), ("gate_col_rows", C.c_uint32), ("lookup_col_rows", C.c_uint32),
                ("spread_rows", C.c_uint32), ("device", C.c_int32), ("build_shape", C.c_uint32), ("block_parts", C.c_uint32),
                ("num_lookup_advice", C.c_uint32)]


class _Layout(C.Structure):
    _fields_ = [("n_digests", C.c_uint32), ("n_gate_cells", C.c_uint32), ("n_lookup_cells", C.c_uint32), ("n_spread_limbs", C.c_uint32),
                ("n_gate_cols", C.c_uint32), ("gate_col_rows", C.c_uint32), ("n_lookup_cols", C.c_uint32), ("lookup_col_rows", C.c_uint32),
                ("n_spread_cols", C.c_uint32), ("spread_rows", C.c_uint32), ("n_blocks", C.c_uint32), ("n_fixed", C.c_uint32),
                ("n_copies", C.c_uint32), ("n_selectors_on", C.c_uint32), ("cells_per_instance", C.c_uint64), ("gate_bytes", C.c_uint64),
                ("lookup_bytes", C.c_uint64), ("spread_bytes", C.c_uint64)]


class _Batch(C.Structure):
    _fields_ = [("n_instances", C.c_uint64), ("msgs", C.c_void_p), ("msgs_on_device", C.c_int32), ("msgs_bytes", C.c_uint64),
                ("offsets", C.c_void_p), ("lens", C.c_void_p), ("precomputed_lens", C.c_void_p), ("gate", C.c_void_p), ("lookup", C.c_void_p),
                ("spread", C.c_void_p), ("digests_dev", C.c_void_p), ("checksums_dev", C.c_void_p), ("digests_host", C.c_void_p),
                ("checksums_host", C.c_void_p), ("stream", C.c_void_p), ("reuse_inputs", C.c_int32), ("time_kernels", C.c_int32),
                ("only_digest", C.c_uint32), ("lookup_mult_dev", C.c_void_p), ("mult_usable_rows", C.c_uint32), ("mult_not_in_table_dev", C.c_void_p),
                ("compact_dict", C.c_void_p), ("keep_lookup_raw", C.c_uint32)]


# column kinds of a permutation column list (h2sha_perm_desc_t; numbered like chip::ColumnKind, instance is new)
COL_GATE, COL_LOOKUP, COL_DENSE, COL_SPREAD, COL_FIXED, COL_INSTANCE = 0, 1, 2, 3, 4, 6


class _PermDesc(C.Structure):
    _fields_ = [("n_columns", C.c_uint32), ("columns", C.c_void_p), ("num_fixed", C.c_uint32), ("columns_per_chunk", C.c_uint32),
                ("bind_output_bytes", C.c_uint32), ("k", C.c_uint32)]


class _CompactInfo(C.Structure):
    _fields_ = [("dict_cells_per_instance", C.c_uint64), ("dict_bytes_per_instance", C.c_uint64), ("cells_per_instance", C.c_uint64), ("n_consts", C.c_uint32)]


class _CheckSite(C.Structure):
    _fields_ = [("n_cells", C.c_uint32), ("kind", C.c_uint32 * 4), ("index", C.c_uint32 * 4), ("row", C.c_uint32 * 4)]


# the classes of the constraint check, in the order of its counters (h2sha_check_batch)
CHECK_CLASSES = ("gates", "copies", "range_lookups", "spread_lookups", "digest_bytes")
CHECK_NONE = 0xFFFFFFFF   # first failing item of a class without a failure


class _LookupInfo(C.Structure):
    _fields_ = [("n_range_lookups", C.c_uint32), ("n_spread_lookups", C.c_uint32), ("range_table_rows", C.c_uint32),
                ("spread_table_rows", C.c_uint32), ("min_usable_rows", C.c_uint32), ("mult_words_per_instance", C.c_uint64)]


_lib = None
_OLD_OK = bool(os.environ.get("TUNE_LIB"))   # tools/tune.py A/B runs load the library of an earlier revision, which lacks the newer entry points


def load_library():
    """dlopen the in-tree engine; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: build it with `python __graft_entry__.py` (nvcc, sm_100a). There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)

    def sig(name, argtypes=None, restype=None):
        f = getattr(L, name, None)
        if f is None:
            if _OLD_OK:   # an earlier revision's library (A/B timing): it simply lacks the newer entry points
                return
            raise ImportError(f"{LIB_PATH} does not export {name}: rebuild it (python __graft_entry__.py)")
        if argtypes is not None:
            f.argtypes = argtypes
        if restype is not None:
            f.restype = restype

    sig("h2sha_create", [C.POINTER(_Config), C.POINTER(C.c_void_p)], C.c_int)
    sig("h2sha_destroy", [C.c_void_p])
    sig("h2sha_last_error", None, C.c_char_p)
    sig("h2sha_get_layout", [C.c_void_p, C.POINTER(_Layout)])
    sig("h2sha_get_breaks", [C.c_void_p, C.c_void_p])
    sig("h2sha_get_handles", [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p])
    sig("h2sha_get_digest_ranges", [C.c_void_p, C.c_void_p])
    sig("h2sha_get_shape", [C.c_void_p] + [C.c_void_p] * 6)
    sig("h2sha_get_lookup_tables", [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)])
    sig("h2sha_digest_batch", [C.c_void_p, C.POINTER(_Batch)])
    sig("h2sha_export_instance", [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p), C.c_uint32, C.c_void_p])
    sig("h2sha_export_batch", [C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_void_p])
    sig("h2sha_get_compact_info", [C.c_void_p, C.POINTER(_CompactInfo)])
    sig("h2sha_get_compact_map", [C.c_void_p] + [C.c_void_p] * 5)
    sig("h2sha_expand_compact", [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.c_int, C.c_uint32])
    sig("h2sha_get_lookup_info", [C.c_void_p, C.POINTER(_LookupInfo)])
    sig("h2sha_lookup_multiplicities", [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p])
    sig("h2sha_permute_lookup", [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p])
    sig("h2sha_permute_lookup_from_raw", [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p])
    sig("h2sha_lookup_product", [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p])
    sig("h2sha_get_permutation", [C.c_void_p, C.POINTER(_PermDesc), C.c_uint32, C.c_void_p])
    sig("h2sha_permutation_product", [C.c_void_p, C.c_uint64, C.POINTER(_PermDesc), C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p])
    sig("h2sha_permute_lookup_per_instance", [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.c_void_p])
    sig("h2sha_permute_lookup_from_raw_per_instance", [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                                       C.c_void_p, C.c_void_p])
    sig("h2sha_lookup_product_per_instance", [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p,
                                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p])
    sig("h2sha_permutation_product_per_instance", [C.c_void_p, C.c_uint64, C.POINTER(_PermDesc), C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p])
    sig("h2sha_check_batch", [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p])
    sig("h2sha_check_batch_per_instance", [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p])
    sig("h2sha_check_site", [C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(_CheckSite)])
    sig("h2sha_gather", [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p])
    sig("h2sha_zero_outputs", [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p])
    sig("h2sha_debug_mont_from_u64", [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p])
    sig("h2sha_debug_mont_from_u32", [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p])
    sig("h2sha_debug_store_probe", [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p])
    sig("h2sha_debug_int_probe", [C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint64), C.c_void_p])
    sig("h2sha_last_launch_count", [C.c_void_p])
    sig("h2sha_last_kernel_ms", [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float)])
    _lib = L
    return L


def _check(rc: int):
    if rc != H2SHA_OK:
        msg = load_library().h2sha_last_error().decode()
        raise (ReferencePanic if rc == H2SHA_EPANIC else EngineError)(rc, msg)


@dataclass
class Layout:
    n_digests: int
    n_gate_cells: int
    n_lookup_cells: int
    n_spread_limbs: int
    n_gate_cols: int
    gate_col_rows: int
    n_lookup_cols: int
    lookup_col_rows: int
    n_spread_cols: int
    spread_rows: int
    n_blocks: int
    n_fixed: int
    n_copies: int
    n_selectors_on: int
    cells_per_instance: int
    gate_bytes: int
    lookup_bytes: int
    spread_bytes: int

    @property
    def bytes_per_instance(self) -> int:
        return self.gate_bytes + self.lookup_bytes + self.spread_bytes


@dataclass
class Shape:
    selectors: np.ndarray        # [n_gate] u8
    copies: np.ndarray           # [n_copies,4] u32
    fixed: np.ndarray            # [n_fixed,4] u64 canonical
    lookup_src: np.ndarray       # [n_lookup] u32
    limb_dense_src: np.ndarray   # [n_limb] u32
    limb_spread_src: np.ndarray  # [n_limb] u32


@dataclass
class AssignedHashResult:
    """lib.rs:31-36: handles are gate-stream indices (map to (column,row) with `Sha256DynamicConfig.cell_position`)."""
    input_len: int
    input_bytes: np.ndarray
    output_bytes: np.ndarray


@dataclass
class BatchResult:
    digests: Optional[np.ndarray]      # [n_msgs,32] u8 (host) when requested
    checksums: Optional[np.ndarray]    # [n_inst,4] u64 (host) when requested
    gate: object = None                # torch tensors [n_inst, cols, rows, 4] int64 (device) when requested
    lookup: object = None
    spread: object = None


def pack_messages(instances: Sequence[Sequence[bytes]]) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """[[msg_d0, msg_d1, ...] per instance] -> (blob u8, offsets u64, lens u32)."""
    flat = [bytes(m) for inst in instances for m in inst]
    lens = np.array([len(m) for m in flat], dtype=np.uint32)
    offs = np.zeros(len(flat), dtype=np.uint64)
    if len(flat) > 1:
        offs[1:] = np.cumsum(lens[:-1], dtype=np.uint64)
    blob = np.frombuffer(b"".join(flat), dtype=np.uint8).copy() if lens.sum() else np.zeros(0, dtype=np.uint8)
    return blob, offs, lens


class Sha256DynamicConfig:
    """Mirror of the reference's `Sha256DynamicConfig<F>` (lib.rs:38-45) for F = bn256::Fr, batch-oriented."""

    ONE_ROUND_INPUT_BYTES = 64  # lib.rs:48

    def __init__(self, handle, max_variable_byte_sizes, device):
        self._h = handle
        self.max_variable_byte_sizes = list(max_variable_byte_sizes)
        self.device = device
        self._layout = None

    # lib.rs:49-69 (+ RangeConfig::configure's lookup_bits / k -> max_rows, lib.rs:409-418)
    @classmethod
    def configure(cls, max_variable_byte_sizes: Sequence[int], *, max_rows: int = (1 << 17) - 9, lookup_bits: int = 16,
                  num_bits_lookup: int = 8, num_advice_columns: int = 2, is_input_range_check: bool = True, device: int = 0,
                  build_shape: bool = False, gate_col_rows: int = 0, lookup_col_rows: int = 0, spread_rows: int = 0,
                  block_parts: int = 0, num_lookup_advice: int = 0) -> "Sha256DynamicConfig":
        L = load_library()
        sizes = (C.c_uint32 * len(max_variable_byte_sizes))(*max_variable_byte_sizes)
        cfg = _Config(len(max_variable_byte_sizes), sizes, max_rows, lookup_bits, num_bits_lookup, num_advice_columns,
                      1 if is_input_range_check else 0, gate_col_rows, lookup_col_rows, spread_rows, device, 1 if build_shape else 0, block_parts,
                      num_lookup_advice)
        h = C.c_void_p()
        _check(L.h2sha_create(C.byref(cfg), C.byref(h)))
        return cls(h, max_variable_byte_sizes, device)

    def close(self):
        if self._h:
            load_library().h2sha_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def layout(self) -> Layout:
        if self._layout is None:
            l = _Layout()
            _check(load_library().h2sha_get_layout(self._h, C.byref(l)))
            self._layout = Layout(*[int(getattr(l, f[0])) for f in _Layout._fields_])
        return self._layout

    def breaks(self) -> np.ndarray:
        b = np.zeros(self.layout.n_gate_cols, dtype=np.uint32)
        _check(load_library().h2sha_get_breaks(self._h, b.ctypes.data_as(C.c_void_p)))
        return b

    def cell_position(self, stream_idx):
        """gate-stream index -> (column, row)."""
        b = self.breaks()
        col = np.searchsorted(b, stream_idx, side="right") - 1
        return col, np.asarray(stream_idx) - b[col]

    def handles(self, d: int = 0) -> AssignedHashResult:
        il = C.c_uint32()
        ib = np.zeros(self.max_variable_byte_sizes[d], dtype=np.uint32)
        ob = np.zeros(32, dtype=np.uint32)
        _check(load_library().h2sha_get_handles(self._h, d, C.byref(il), ib.ctypes.data_as(C.c_void_p), ob.ctypes.data_as(C.c_void_p)))
        return AssignedHashResult(int(il.value), ib, ob)

    def digest_ranges(self) -> np.ndarray:
        """[n_digests, 6]: gate_lo, gate_hi, lookup_lo, lookup_hi, limb_lo, limb_hi of the stream ranges each digest() call owns."""
        r = np.zeros((len(self.max_variable_byte_sizes), 6), dtype=np.uint32)
        _check(load_library().h2sha_get_digest_ranges(self._h, r.ctypes.data_as(C.c_void_p)))
        return r

    def shape(self) -> Shape:
        lay = self.layout
        sel = np.zeros(lay.n_gate_cells, dtype=np.uint8)
        cp = np.zeros((lay.n_copies, 4), dtype=np.uint32)
        fx = np.zeros((lay.n_fixed, 4), dtype=np.uint64)
        ls = np.zeros(lay.n_lookup_cells, dtype=np.uint32)
        ld = np.zeros(lay.n_spread_limbs, dtype=np.uint32)
        lsp = np.zeros(lay.n_spread_limbs, dtype=np.uint32)
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        _check(load_library().h2sha_get_shape(self._h, p(sel), p(cp), p(fx), p(ls), p(ld), p(lsp)))
        return Shape(sel, cp, fx, ls, ld, lsp)

    def store_probe(self, buf_ptr: int, nbytes: int, stream: int = 0):
        """Measurement hook: plain coalesced 256-bit stores of incompressible cells over [buf_ptr, buf_ptr + nbytes)."""
        _check(load_library().h2sha_debug_store_probe(self._h, C.c_void_p(buf_ptr), C.c_uint64(nbytes), C.c_void_p(stream)))

    def int_probe(self, scratch_ptr: int, iters: int, stream: int = 0) -> int:
        """Measurement hook: IMAD/LOP3 dependency chains, no memory traffic; returns the integer instructions the launch executes."""
        n = C.c_uint64()
        _check(load_library().h2sha_debug_int_probe(self._h, C.c_void_p(scratch_ptr), C.c_uint32(iters), C.byref(n), C.c_void_p(stream)))
        return int(n.value)

    def lookup_tables(self):
        """(dense[2^bits], spread[2^bits], n_range_rows): SpreadConfig::load (spread.rs:165-194) and the range table's row count."""
        L = load_library()
        ns, nr = C.c_uint32(), C.c_uint32()
        _check(L.h2sha_get_lookup_tables(self._h, None, None, C.byref(ns), C.byref(nr)))
        d = np.zeros(ns.value, dtype=np.uint64); sp = np.zeros(ns.value, dtype=np.uint64)
        _check(L.h2sha_get_lookup_tables(self._h, d.ctypes.data_as(C.c_void_p), sp.ctypes.data_as(C.c_void_p), C.byref(ns), C.byref(nr)))
        return d, sp, int(nr.value)

    # ------------------------------------------------------------------------------------------------
    def alloc_outputs(self, n_instances: int, zero: bool = True):
        """Device buffers [n_inst, cols, rows, 4] int64 for gate / lookup / spread."""
        import torch
        lay = self.layout
        dev = torch.device("cuda", self.device)
        mk = (torch.zeros if zero else torch.empty)
        gate = mk((n_instances, lay.n_gate_cols, lay.gate_col_rows, 4), dtype=torch.int64, device=dev)
        lookup = mk((n_instances, lay.n_lookup_cols, lay.lookup_col_rows, 4), dtype=torch.int64, device=dev)
        spread = mk((n_instances, lay.n_spread_cols, lay.spread_rows, 4), dtype=torch.int64, device=dev)
        return gate, lookup, spread

    def digest_batch_raw(self, n_instances: int, msgs_ptr: int, msgs_on_device: bool, msgs_bytes: int, offsets: np.ndarray, lens: np.ndarray,
                         precomputed_lens: Optional[np.ndarray], *, gate_ptr: int = 0, lookup_ptr: int = 0, spread_ptr: int = 0,
                         digests_dev_ptr: int = 0, checksums_dev_ptr: int = 0, digests_host_ptr: int = 0, checksums_host_ptr: int = 0,
                         stream: int = 0, reuse_inputs: bool = False, time_kernels: bool = False, only_digest: int = 0,
                         lookup_mult_ptr: int = 0, mult_usable_rows: int = 0, mult_bad_ptr: int = 0, compact_dict_ptr: int = 0,
                         keep_lookup_raw: bool = False):
        """Thin wrapper over h2sha_digest_batch (all pointers are integers)."""
        if reuse_inputs:
            off_p = len_p = pre_p = None
        else:
            assert offsets.dtype == np.uint64 and lens.dtype == np.uint32
            off_p, len_p = offsets.ctypes.data, lens.ctypes.data
            pre_p = precomputed_lens.ctypes.data if precomputed_lens is not None else None
        b = _Batch(n_instances, msgs_ptr or None, 1 if msgs_on_device else 0, msgs_bytes, off_p, len_p, pre_p, gate_ptr or None,
                   lookup_ptr or None, spread_ptr or None, digests_dev_ptr or None, checksums_dev_ptr or None, digests_host_ptr or None,
                   checksums_host_ptr or None, stream or None, 1 if reuse_inputs else 0, 1 if time_kernels else 0, only_digest,
                   lookup_mult_ptr or None, mult_usable_rows, mult_bad_ptr or None, compact_dict_ptr or None, 1 if keep_lookup_raw else 0)
        _check(load_library().h2sha_digest_batch(self._h, C.byref(b)))

    def last_kernel_ms(self) -> Tuple[float, float]:
        """(k_trace ms, k_expand ms) of the last batch run with time_kernels=True."""
        a, b = C.c_float(), C.c_float()
        _check(load_library().h2sha_last_kernel_ms(self._h, C.byref(a), C.byref(b)))
        return float(a.value), float(b.value)

    def digest_batch(self, instances: Sequence[Sequence[bytes]], precomputed_input_lens: Optional[Sequence[Sequence[int]]] = None, *,
                     want_cells: bool = True, outputs=None) -> BatchResult:
        """digest() (lib.rs:71-349) for every message of every instance.  instances[i][d] is the input of the d-th
        digest call of instance i; precomputed_input_lens[i][d] its `precomputed_input_len` (None = no prefix)."""
        import torch
        if self.device < 0:
            raise EngineError(H2SHA_ECUDA, "plan-only engine (device=-1): witness generation needs a CUDA device; there is no CPU path")
        D = len(self.max_variable_byte_sizes)
        n = len(instances)
        for inst in instances:
            if len(inst) != D:
                raise EngineError(H2SHA_EINVAL, f"each instance needs {D} messages")
        blob, offs, lens = pack_messages(instances)
        pre = None
        if precomputed_input_lens is not None:
            pre = np.array([p for inst in precomputed_input_lens for p in inst], dtype=np.uint32)
        digests = np.zeros((n * D, 32), dtype=np.uint8)
        cks = np.zeros((n, 4), dtype=np.uint64)
        gate = lookup = spread = None
        if want_cells:
            gate, lookup, spread = outputs if outputs is not None else self.alloc_outputs(n)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        self.digest_batch_raw(n, blob.ctypes.data if blob.size else 0, False, int(blob.size), offs, lens, pre,
                              gate_ptr=gate.data_ptr() if gate is not None else 0, lookup_ptr=lookup.data_ptr() if lookup is not None else 0,
                              spread_ptr=spread.data_ptr() if spread is not None else 0, digests_host_ptr=digests.ctypes.data,
                              checksums_host_ptr=cks.ctypes.data, stream=stream)
        torch.cuda.current_stream(self.device).synchronize()
        return BatchResult(digests, cks, gate, lookup, spread)

    def digest(self, input: bytes, precomputed_input_len: Optional[int] = None) -> Tuple[AssignedHashResult, BatchResult]:
        """Single-message convenience with the reference's signature (only for n_digests == 1 configurations)."""
        if len(self.max_variable_byte_sizes) != 1:
            raise EngineError(H2SHA_EINVAL, "digest() needs a single-digest configuration; use digest_batch")
        res = self.digest_batch([[input]], [[precomputed_input_len or 0]] if precomputed_input_len is not None else None)
        return self.handles(0), res

    def export_instance(self, res: "BatchResult", instance: int, rows_per_column: int) -> np.ndarray:
        """Prover hand-off: the advice columns of one instance as a host array [n_columns, rows_per_column, 4] u64
        (gate columns, lookup column(s), dense_0.., spread_0..), zero-padded like halo2's witness vectors."""
        import torch
        lay = self.layout
        n_cols = lay.n_gate_cols + lay.n_lookup_cols + lay.n_spread_cols
        out = np.zeros((n_cols, rows_per_column, 4), dtype=np.uint64)
        ptrs = (C.c_void_p * n_cols)(*[out[c].ctypes.data for c in range(n_cols)])
        _check(load_library().h2sha_export_instance(self._h, instance, res.gate.data_ptr(), res.lookup.data_ptr(), res.spread.data_ptr(), ptrs,
                                                    rows_per_column, torch.cuda.current_stream(self.device).cuda_stream))
        torch.cuda.current_stream(self.device).synchronize()
        return out

    # ---- prover hand-off of whole batches ----
    def n_columns(self) -> int:
        lay = self.layout
        return lay.n_gate_cols + lay.n_lookup_cols + lay.n_spread_cols

    def export_batch(self, res: "BatchResult", first: int, n: int, rows_per_column: int, out=None):
        """Instances [first, first+n) of a batch as a pinned host tensor [n, n_columns, rows_per_column, 4] int64 (zero-padded columns in
        the reference's allocation order): three strided D2H copies for the whole range."""
        import torch
        if out is None:
            out = torch.zeros((n, self.n_columns(), rows_per_column, 4), dtype=torch.int64).pin_memory()
        _check(load_library().h2sha_export_batch(self._h, first, n, res.gate.data_ptr(), res.lookup.data_ptr(), res.spread.data_ptr(), out.data_ptr(),
                                                 rows_per_column, 0, torch.cuda.current_stream(self.device).cuda_stream))
        torch.cuda.current_stream(self.device).synchronize()
        return out

    def compact_info(self) -> dict:
        ci = _CompactInfo()
        _check(load_library().h2sha_get_compact_info(self._h, C.byref(ci)))
        return {f[0]: int(getattr(ci, f[0])) for f in _CompactInfo._fields_}

    def compact_map(self):
        """(gate_map, lookup_map, dense_map, spread_map, consts): which dictionary entry (or 0x80000000 | constant index) each cell copies."""
        lay, ci = self.layout, self.compact_info()
        g = np.zeros(lay.n_gate_cells, np.uint32); l = np.zeros(lay.n_lookup_cells, np.uint32)
        d = np.zeros(lay.n_spread_limbs, np.uint32); s = np.zeros(lay.n_spread_limbs, np.uint32)
        c = np.zeros((ci["n_consts"], 4), np.uint64)
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        _check(load_library().h2sha_get_compact_map(self._h, p(g), p(l), p(d), p(s), p(c)))
        return g, l, d, s, c

    def expand_compact(self, dict_host, n: int, rows_per_column: int, out=None, n_threads: int = 0, zero_fill: bool = True):
        """Host-side expander of the compact hand-off: dictionary [n, dict_cells, 4] (numpy or CPU tensor) -> [n, n_columns, rows_per_column, 4]."""
        dptr = dict_host.ctypes.data if isinstance(dict_host, np.ndarray) else dict_host.data_ptr()
        if out is None:
            out = np.empty((n, self.n_columns(), rows_per_column, 4), dtype=np.uint64)
        optr = out.ctypes.data if isinstance(out, np.ndarray) else out.data_ptr()
        _check(load_library().h2sha_expand_compact(self._h, C.c_void_p(dptr), n, C.c_void_p(optr), rows_per_column, 1 if zero_fill else 0, n_threads))
        return out

    def check_batch(self, res: "BatchResult", digests_dev_ptr: int = 0) -> dict:
        """MockProver-style check of every instance of a batch on the device (gates, copies, lookups, digest bytes):
        violation counts, all zero for a witness the reference's tests would accept (lib.rs:525-526)."""
        import torch
        v = np.zeros(5, dtype=np.uint64)
        _check(load_library().h2sha_check_batch(self._h, res.gate.shape[0], res.gate.data_ptr(), res.lookup.data_ptr(), res.spread.data_ptr(),
                                                C.c_void_p(digests_dev_ptr or None), v.ctypes.data_as(C.c_void_p),
                                                torch.cuda.current_stream(self.device).cuda_stream))
        return dict(zip(CHECK_CLASSES, (int(x) for x in v)))

    def check_batch_per_instance(self, res: "BatchResult", digests_dev_ptr: int = 0) -> Tuple[np.ndarray, np.ndarray]:
        """The same check with a verdict per instance: (counts, first), numpy u32 [n_instances, 5] in the order of CHECK_CLASSES.
        first[i, c] is the smallest failing item number of class c in instance i (CHECK_NONE when none fails); check_site names its cells."""
        import torch
        n = res.gate.shape[0]
        out = torch.empty((2, n, 5), dtype=torch.int32, device=torch.device("cuda", self.device))
        _check(load_library().h2sha_check_batch_per_instance(self._h, n, res.gate.data_ptr(), res.lookup.data_ptr(), res.spread.data_ptr(),
                                                             C.c_void_p(digests_dev_ptr or None), out[0].data_ptr(), out[1].data_ptr(),
                                                             torch.cuda.current_stream(self.device).cuda_stream))
        o = out.cpu().numpy().view(np.uint32)
        return o[0], o[1]

    def check_site(self, cls: int, item: int) -> dict:
        """The cells check item `item` of class `cls` reads: {"kind", "index", "row"} lists (kinds COL_*; rows from the region's row 0)."""
        s = _CheckSite()
        _check(load_library().h2sha_check_site(self._h, cls, item, C.byref(s)))
        n = s.n_cells
        return dict(kind=list(s.kind[:n]), index=list(s.index[:n]), row=list(s.row[:n]))

    # ---- lookup-argument pre-work (halo2 lookup prover `permute_expression_pair`; spread.rs:53-62, lib.rs:409-418,469) ----
    def lookup_info(self) -> dict:
        li = _LookupInfo()
        _check(load_library().h2sha_get_lookup_info(self._h, C.byref(li)))
        return {f[0]: int(getattr(li, f[0])) for f in _LookupInfo._fields_}

    def lookup_multiplicities(self, res: "BatchResult", usable_rows: int):
        """(mult [n_inst, mult_words_per_instance] int32 device tensor, cells that are no table row) of a batch's witness."""
        import torch
        n = res.lookup.shape[0]
        info = self.lookup_info()
        dev = torch.device("cuda", self.device)
        mult = torch.empty((n, info["mult_words_per_instance"]), dtype=torch.int32, device=dev)
        bad = torch.zeros(1, dtype=torch.int32, device=dev)
        _check(load_library().h2sha_lookup_multiplicities(self._h, n, res.lookup.data_ptr(), res.spread.data_ptr(), usable_rows, mult.data_ptr(),
                                                          bad.data_ptr(), torch.cuda.current_stream(self.device).cuda_stream))
        return mult, int(bad.item())

    def permute_lookup(self, mult, lookup_idx: int, usable_rows: int, theta_mont: Optional[np.ndarray] = None):
        """(A', S') of lookup `lookup_idx` for every instance: device tensors [n_inst, usable_rows, 4] int64 (Montgomery Fr)."""
        import torch
        n = mult.shape[0]
        dev = torch.device("cuda", self.device)
        a = torch.empty((n, usable_rows, 4), dtype=torch.int64, device=dev)
        s = torch.empty((n, usable_rows, 4), dtype=torch.int64, device=dev)
        err = torch.zeros(1, dtype=torch.int32, device=dev)
        th = None
        if theta_mont is not None:
            th = np.ascontiguousarray(theta_mont, dtype=np.uint64)
            assert th.shape == (4,)
        _check(load_library().h2sha_permute_lookup(self._h, n, lookup_idx, mult.data_ptr(), usable_rows, th.ctypes.data if th is not None else None,
                                                   a.data_ptr(), s.data_ptr(), err.data_ptr(), torch.cuda.current_stream(self.device).cuda_stream))
        if int(err.item()):
            raise EngineError(H2SHA_EINVAL, f"{int(err.item())} instance(s) whose multiplicities do not cover usable_rows")
        return a, s

    def permute_lookup_from_raw(self, first_instance: int, n_instances: int, lookup_idx: int, usable_rows: int, theta_mont: Optional[np.ndarray] = None):
        """(A', S') like permute_lookup, from the raw value lists the last keep_lookup_raw / lookup_mult batch left in the engine."""
        import torch
        dev = torch.device("cuda", self.device)
        a = torch.empty((n_instances, usable_rows, 4), dtype=torch.int64, device=dev)
        s = torch.empty((n_instances, usable_rows, 4), dtype=torch.int64, device=dev)
        err = torch.zeros(1, dtype=torch.int32, device=dev)
        th = None
        if theta_mont is not None:
            th = np.ascontiguousarray(theta_mont, dtype=np.uint64)
            assert th.shape == (4,)
        _check(load_library().h2sha_permute_lookup_from_raw(self._h, first_instance, n_instances, lookup_idx, usable_rows, th.ctypes.data if th is not None else None,
                                                            a.data_ptr(), s.data_ptr(), err.data_ptr(), torch.cuda.current_stream(self.device).cuda_stream))
        if int(err.item()):
            raise EngineError(H2SHA_EINVAL, f"{int(err.item())} instance(s) whose multiplicities do not cover usable_rows")
        return a, s

    def lookup_product(self, res: "BatchResult", lookup_idx: int, a_p, s_p, usable_rows: int, beta_mont: np.ndarray, gamma_mont: np.ndarray,
                       theta_mont: Optional[np.ndarray] = None):
        """(z [n_inst, usable_rows + 1, 4] int64 device tensor, instances whose z[usable_rows] != 1) of lookup `lookup_idx`, halo2's
        `commit_product` from the batch's witness `res` and the permuted pair (A', S') [n_inst, usable_rows, 4] of the same instances."""
        import torch
        n = a_p.shape[0]
        if tuple(a_p.shape) != (n, usable_rows, 4) or tuple(s_p.shape) != (n, usable_rows, 4):
            raise EngineError(H2SHA_EINVAL, "A' and S' must be [n_instances, usable_rows, 4]")
        for buf in (res.lookup, res.spread):
            if buf is not None and buf.shape[0] < n:
                raise EngineError(H2SHA_EINVAL, "the witness holds fewer instances than A' and S'")
        dev = torch.device("cuda", self.device)
        z = torch.empty((n, usable_rows + 1, 4), dtype=torch.int64, device=dev)
        err = torch.zeros(1, dtype=torch.int32, device=dev)
        ch = [None if x is None else np.ascontiguousarray(x, dtype=np.uint64) for x in (theta_mont, beta_mont, gamma_mont)]
        assert all(x is None or x.shape == (4,) for x in ch)
        ptr = lambda t: t.data_ptr() if t is not None else None
        _check(load_library().h2sha_lookup_product(self._h, n, lookup_idx, ptr(res.lookup), ptr(res.spread), a_p.data_ptr(), s_p.data_ptr(), usable_rows,
                                                   *[x.ctypes.data if x is not None else None for x in ch], z.data_ptr(), err.data_ptr(),
                                                   torch.cuda.current_stream(self.device).cuda_stream))
        return z, int(err.item())

    # ---- permutation argument (halo2 plonk/permutation: keygen Assembly, prover `Argument::commit`) ----
    @staticmethod
    def _perm_desc(columns, num_fixed: int, columns_per_chunk: int, bind_output_bytes: bool, k: int):
        cols = np.ascontiguousarray(np.asarray(columns, dtype=np.uint32).reshape(-1, 2))
        return _PermDesc(len(cols), cols.ctypes.data, num_fixed, columns_per_chunk, 1 if bind_output_bytes else 0, k), cols

    def permutation_mapping(self, columns, usable_rows: int, *, columns_per_chunk: int, num_fixed: int = 1, bind_output_bytes: bool = False,
                            k: int = 0) -> np.ndarray:
        """halo2 keygen `Assembly` mapping of the chip's copy constraints: [len(columns), usable_rows, 2] u32 (column position, row).
        `columns`: (kind, index) pairs (COL_*) in the order of `cs.permutation.columns`.  Works on a plan-only configuration
        (device=-1, build_shape=True)."""
        d, cols = self._perm_desc(columns, num_fixed, columns_per_chunk, bind_output_bytes, k)
        m = np.zeros((len(cols), usable_rows, 2), dtype=np.uint32)
        _check(load_library().h2sha_get_permutation(self._h, C.byref(d), usable_rows, m.ctypes.data_as(C.c_void_p)))
        return m

    def permutation_product(self, res: "BatchResult", columns, usable_rows: int, beta_mont: np.ndarray, gamma_mont: np.ndarray, *,
                            columns_per_chunk: int, num_fixed: int = 1, bind_output_bytes: bool = False, digests=None, k: int = 0):
        """(z [n_inst, n_chunks, usable_rows + 1, 4] int64 device tensor, instances whose last z[usable_rows] != 1): the permutation
        argument's product columns (halo2 `permutation::prover` commit) of a batch's witness `res`.  `digests` ([n_msgs, 32] u8, host
        array or device tensor) fills the instance column; needed only with bind_output_bytes."""
        import torch
        n = res.gate.shape[0]
        for buf in (res.lookup, res.spread):
            if buf is not None and buf.shape[0] < n:
                raise EngineError(H2SHA_EINVAL, "the witness buffers hold different numbers of instances")
        d, cols = self._perm_desc(columns, num_fixed, columns_per_chunk, bind_output_bytes, k)
        dev = torch.device("cuda", self.device)
        n_chunks = -(-len(cols) // columns_per_chunk) if columns_per_chunk else 0
        z = torch.empty((n, n_chunks, usable_rows + 1, 4), dtype=torch.int64, device=dev)
        err = torch.zeros(1, dtype=torch.int32, device=dev)
        dg = None
        if digests is not None:
            dg = digests if isinstance(digests, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(digests, dtype=np.uint8))
            dg = dg.to(dev).contiguous()
            if dg.numel() < n * 32 * len(self.max_variable_byte_sizes):
                raise EngineError(H2SHA_EINVAL, "digests holds fewer messages than the batch")
        bg = [np.ascontiguousarray(x, dtype=np.uint64) for x in (beta_mont, gamma_mont)]
        assert all(x.shape == (4,) for x in bg)
        ptr = lambda t: t.data_ptr() if t is not None else None
        _check(load_library().h2sha_permutation_product(self._h, n, C.byref(d), usable_rows, ptr(res.gate), ptr(res.lookup), ptr(res.spread), ptr(dg),
                                                        bg[0].ctypes.data, bg[1].ctypes.data, z.data_ptr(), err.data_ptr(),
                                                        torch.cuda.current_stream(self.device).cuda_stream))
        return z, int(err.item())

    # ---- per-instance challenges: one (theta_i, beta_i, gamma_i) per instance, for batches of independent proofs ----
    @staticmethod
    def _challenge_rows(x, n: int, name: str):
        """[n, 4] u64 host array (Montgomery) of one challenge per instance, or None."""
        if x is None:
            return None
        a = np.ascontiguousarray(x, dtype=np.uint64)
        if a.shape != (n, 4):
            raise EngineError(H2SHA_EINVAL, f"{name} must be [n_instances, 4] u64, not {list(a.shape)}")
        return a

    def _per_instance_errors(self, n: int):
        import torch
        return torch.zeros(n, dtype=torch.int32, device=torch.device("cuda", self.device))

    def permute_lookup_per_instance(self, mult, lookup_idx: int, usable_rows: int, thetas=None):
        """(A', S', errors) like permute_lookup with theta_i of instance i (`thetas` [n, 4] u64 Montgomery; None for a range lookup).
        errors [n] int numpy: instance i's multiplicities do not cover usable_rows, or theta_i makes two spread-table rows equal
        (its A', S' rows are then left unwritten).  Never raises for such per-instance failures."""
        import torch
        n = mult.shape[0]
        th = self._challenge_rows(thetas, n, "thetas")
        dev = torch.device("cuda", self.device)
        a = torch.empty((n, usable_rows, 4), dtype=torch.int64, device=dev)
        s = torch.empty((n, usable_rows, 4), dtype=torch.int64, device=dev)
        err = self._per_instance_errors(n)
        _check(load_library().h2sha_permute_lookup_per_instance(self._h, n, lookup_idx, mult.data_ptr(), usable_rows, th.ctypes.data if th is not None else None,
                                                                a.data_ptr(), s.data_ptr(), err.data_ptr(), torch.cuda.current_stream(self.device).cuda_stream))
        return a, s, err.cpu().numpy()

    def permute_lookup_from_raw_per_instance(self, first_instance: int, n_instances: int, lookup_idx: int, usable_rows: int, thetas=None):
        """(A', S', errors) like permute_lookup_per_instance, from the raw value lists the last keep_lookup_raw / lookup_mult batch left in
        the engine; row i of `thetas` belongs to instance first_instance + i."""
        import torch
        th = self._challenge_rows(thetas, n_instances, "thetas")
        dev = torch.device("cuda", self.device)
        a = torch.empty((n_instances, usable_rows, 4), dtype=torch.int64, device=dev)
        s = torch.empty((n_instances, usable_rows, 4), dtype=torch.int64, device=dev)
        err = self._per_instance_errors(n_instances)
        _check(load_library().h2sha_permute_lookup_from_raw_per_instance(self._h, first_instance, n_instances, lookup_idx, usable_rows,
                                                                         th.ctypes.data if th is not None else None, a.data_ptr(), s.data_ptr(),
                                                                         err.data_ptr(), torch.cuda.current_stream(self.device).cuda_stream))
        return a, s, err.cpu().numpy()

    def lookup_product_per_instance(self, res: "BatchResult", lookup_idx: int, a_p, s_p, usable_rows: int, betas, gammas, thetas=None):
        """(z, errors) like lookup_product with theta_i, beta_i, gamma_i of instance i ([n, 4] u64 Montgomery each; thetas only for a
        spread lookup).  errors [n] int numpy: instance i's z[usable_rows] != 1."""
        import torch
        n = a_p.shape[0]
        if tuple(a_p.shape) != (n, usable_rows, 4) or tuple(s_p.shape) != (n, usable_rows, 4):
            raise EngineError(H2SHA_EINVAL, "A' and S' must be [n_instances, usable_rows, 4]")
        for buf in (res.lookup, res.spread):
            if buf is not None and buf.shape[0] < n:
                raise EngineError(H2SHA_EINVAL, "the witness holds fewer instances than A' and S'")
        ch = [self._challenge_rows(x, n, name) for x, name in ((thetas, "thetas"), (betas, "betas"), (gammas, "gammas"))]
        dev = torch.device("cuda", self.device)
        z = torch.empty((n, usable_rows + 1, 4), dtype=torch.int64, device=dev)
        err = self._per_instance_errors(n)
        ptr = lambda t: t.data_ptr() if t is not None else None
        _check(load_library().h2sha_lookup_product_per_instance(self._h, n, lookup_idx, ptr(res.lookup), ptr(res.spread), a_p.data_ptr(), s_p.data_ptr(),
                                                                usable_rows, *[x.ctypes.data if x is not None else None for x in ch], z.data_ptr(),
                                                                err.data_ptr(), torch.cuda.current_stream(self.device).cuda_stream))
        return z, err.cpu().numpy()

    def permutation_product_per_instance(self, res: "BatchResult", columns, usable_rows: int, betas, gammas, *, columns_per_chunk: int,
                                         num_fixed: int = 1, bind_output_bytes: bool = False, digests=None, k: int = 0):
        """(z, errors) like permutation_product with beta_i, gamma_i of instance i ([n, 4] u64 Montgomery each).  errors [n] int numpy:
        instance i's last z[usable_rows] != 1."""
        import torch
        n = res.gate.shape[0]
        for buf in (res.lookup, res.spread):
            if buf is not None and buf.shape[0] < n:
                raise EngineError(H2SHA_EINVAL, "the witness buffers hold different numbers of instances")
        bg = [self._challenge_rows(x, n, name) for x, name in ((betas, "betas"), (gammas, "gammas"))]
        d, cols = self._perm_desc(columns, num_fixed, columns_per_chunk, bind_output_bytes, k)
        dev = torch.device("cuda", self.device)
        n_chunks = -(-len(cols) // columns_per_chunk) if columns_per_chunk else 0
        z = torch.empty((n, n_chunks, usable_rows + 1, 4), dtype=torch.int64, device=dev)
        err = self._per_instance_errors(n)
        dg = None
        if digests is not None:
            dg = digests if isinstance(digests, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(digests, dtype=np.uint8))
            dg = dg.to(dev).contiguous()
            if dg.numel() < n * 32 * len(self.max_variable_byte_sizes):
                raise EngineError(H2SHA_EINVAL, "digests holds fewer messages than the batch")
        ptr = lambda t: t.data_ptr() if t is not None else None
        _check(load_library().h2sha_permutation_product_per_instance(self._h, n, C.byref(d), usable_rows, ptr(res.gate), ptr(res.lookup), ptr(res.spread),
                                                                     ptr(dg), bg[0].ctypes.data, bg[1].ctypes.data, z.data_ptr(), err.data_ptr(),
                                                                     torch.cuda.current_stream(self.device).cuda_stream))
        return z, err.cpu().numpy()

    def launches_last_batch(self) -> int:
        return int(load_library().h2sha_last_launch_count(self._h))

    def mont_from_u64(self, vals: np.ndarray, path32: bool = False) -> np.ndarray:
        """Test hook: device Montgomery conversion of raw u64 values -> [n,4] u64 (path32: the < 2^32 fast path)."""
        import torch
        dev = torch.device("cuda", self.device)
        v = torch.from_numpy(vals.astype(np.uint64).view(np.int64)).to(dev)
        out = torch.empty((v.numel(), 4), dtype=torch.int64, device=dev)
        fn = load_library().h2sha_debug_mont_from_u32 if path32 else load_library().h2sha_debug_mont_from_u64
        _check(fn(self._h, v.data_ptr(), out.data_ptr(), v.numel(), torch.cuda.current_stream(self.device).cuda_stream))
        torch.cuda.current_stream(self.device).synchronize()
        return out.cpu().numpy().view(np.uint64)
