"""ctypes binding of libxsparse_b200.so -- one Python function per C-ABI entry point of
include/xsparse_b200.h.  There is no fallback: if the shared library is missing or fails
to load, importing this module raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libxsparse_b200.so")

# status codes / enums (include/xsparse_b200.h)
OK, EBOUNDS, ESIZE, EILLEGAL, EINVAL, ECUDA, ENOMEM, ESTATE = range(8)
F64 = 0
I32, I64 = 0, 1
UPDATE, RAW, ASSIGN = 0, 1, 2
# xsb_triplet of include/xsparse_b200.h: what one updateindex! call appends to the host buffer
TRIPLET_DTYPE = np.dtype([("row", "<u4"), ("col", "<u4"), ("val", "<f8")])
assert TRIPLET_DTYPE.itemsize == 16
DETERMINISTIC, FAST = 0, 1
COMBINE_SEED, COMBINE_ADD = 0, 1
STRATEGY_AUTO, STRATEGY_FULLSORT = 0, 1
GROUPING_AUTO, GROUPING_OFF, GROUPING_ON = 0, 1, 2
OP_ADD, OP_SUB = 0, 1


class XsbError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"[xsb {code}] {msg}")
        self.code = code


class XsbBoundsError(XsbError, IndexError):
    """Julia BoundsError (sparsematrixcsc.jl:8-10)."""


class XsbSizeError(XsbError, AssertionError):
    """size-mismatch @assert (sparsematrixlnk.jl:296-297)."""


class XsbIllegalError(XsbError):
    """error(...) of the MT wrapper (genericmtextendablesparsematrixcsc.jl:67,80)."""


class FlushStats(C.Structure):
    _fields_ = [
        ("n_inserted", C.c_int64),
        ("nnz_old", C.c_int64),
        ("nnz_new", C.c_int64),
        ("sort_passes", C.c_int32),
        ("sort_bits", C.c_int32),
        ("kernel_launches", C.c_int32),
        ("column_path", C.c_int32),
        ("ms_total", C.c_float),
        ("ms_expand", C.c_float),
        ("ms_histogram", C.c_float),
        ("ms_sort", C.c_float),
        ("ms_reduce", C.c_float),
        ("ms_colptr", C.c_float),
        ("ms_other", C.c_float),
        ("ms_host_alloc", C.c_float),
        ("group_pairs", C.c_int64),
        ("ms_group_count", C.c_float),
        ("ms_pair_sort", C.c_float),
        ("ms_group_scatter", C.c_float),
        ("ms_fold", C.c_float),
        ("ms_compact", C.c_float),
        ("direct_fold", C.c_int32),
        ("preagg_records", C.c_int64),
        ("ms_preagg", C.c_float),
        ("precounted", C.c_float),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


_i32, _i64, _u64, _p, _f64 = C.c_int32, C.c_int64, C.c_uint64, C.c_void_p, C.c_double

# name -> (restype, argtypes): every symbol include/xsparse_b200.h declares
SIGNATURES = {
    "xsb_version": (_i32, []),
    "xsb_device_count": (_i32, [C.POINTER(_i32)]),
    "xsb_create": (_i32, [_i64, _i64, _i32, _i32, _i32, _i32, _i32, C.POINTER(_p)]),
    "xsb_create_slab": (_i32, [_i64, _i64, _i32, _i32, C.POINTER(_i64), _i32, _i32, _i32, _i32, C.POINTER(_p)]),
    "xsb_slab_info": (_i32, [_p, C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_i64)]),
    "xsb_route_prepare": (_i32, [_p, _p, _i64, C.POINTER(_i64)]),
    "xsb_route_count": (_i32, [_p, C.POINTER(_i64)]),
    "xsb_route_finish": (_i32, [_p, _i32, _p, _i64]),
    "xsb_route_pack": (_i32, [_p, _p, C.POINTER(_i64), _i64]),
    "xsb_route_unpack": (_i32, [_p, _p, C.POINTER(_i64)]),
    "xsb_peer_exchange_create": (_i32, [_p, C.POINTER(_i64), _p]),
    "xsb_peer_exchange_connect": (_i32, [_p, _p]),
    "xsb_peer_exchange_connect_local": (_i32, [_p, C.POINTER(_p)]),
    "xsb_peer_exchange_disconnect": (_i32, [_p]),
    "xsb_peer_exchange_destroy": (_i32, [_p]),
    "xsb_route_pack_peer": (_i32, [_p]),
    "xsb_route_unpack_peer": (_i32, [_p]),
    "xsb_destroy": (_i32, [_p]),
    "xsb_last_error": (C.c_char_p, [_p]),
    "xsb_reset": (_i32, [_p]),
    "xsb_set_csc": (_i32, [_p, _p, _p, _p]),
    "xsb_shrink_to_fit": (_i32, [_p]),
    "xsb_size": (_i32, [_p, C.POINTER(_i64), C.POINTER(_i64)]),
    "xsb_nnz": (_i32, [_p, C.POINTER(_i64)]),
    "xsb_reserve": (_i32, [_p, _i32, _i64]),
    "xsb_insert_batch": (_i32, [_p, _i32, _p, _p, _p, _i64, _i32]),
    "xsb_insert_triplets": (_i32, [_p, _i32, _p, _i64, _i32]),
    "xsb_insert_elements": (_i32, [_p, _i32, _i32, _i64, _p, _p, _i32]),
    "xsb_insert_elements_rect": (_i32, [_p, _i32, _i32, _i32, _i64, _p, _p, _p, _i32]),
    "xsb_pending": (_i32, [_p, C.POINTER(_i64)]),
    "xsb_flush": (_i32, [_p, _i32, C.POINTER(_i64), C.POINTER(_i32)]),
    "xsb_flush_ex": (_i32, [_p, _i32, _i32, C.POINTER(_i64), C.POINTER(_i32)]),
    "xsb_fetch_csc": (_i32, [_p, _p, _p, _p]),
    "xsb_get_values": (_i32, [_p, _p, _p, _p, _i64]),
    "xsb_zero_values": (_i32, [_p]),
    "xsb_freeze_pattern": (_i32, [_p, _p, _p, _i64]),
    "xsb_freeze_elements": (_i32, [_p, _i32, _i64, _p]),
    "xsb_freeze_elements_rect": (_i32, [_p, _i32, _i32, _i64, _p, _p]),
    "xsb_reassemble_values": (_i32, [_p, _p, _i64, _i32]),
    "xsb_reassemble_values_zeroed": (_i32, [_p, _p, _i64, _i32]),
    "xsb_unfreeze": (_i32, [_p]),
    "xsb_freeze_slab": (_i32, [_p, _p, _p, _i64, C.POINTER(_i64)]),
    "xsb_freeze_slab_elements": (_i32, [_p, _i32, _i64, _p, C.POINTER(_i64)]),
    "xsb_freeze_slab_elements_rect": (_i32, [_p, _i32, _i32, _i64, _p, _p, C.POINTER(_i64)]),
    "xsb_freeze_slab_prepare": (_i32, [_p, _p, _i64]),
    "xsb_freeze_slab_finish": (_i32, [_p, _p, C.POINTER(_i64)]),
    "xsb_frozen_slab_counts": (_i32, [_p, C.POINTER(_i64), C.POINTER(_i64)]),
    "xsb_reassemble_slab_pack": (_i32, [_p, _p, _i64, _p]),
    "xsb_reassemble_slab_values": (_i32, [_p, _p, _i64, _p, _i32, _i32]),
    "xsb_mark_dirichlet": (_i32, [_p, _f64, _p]),
    "xsb_eliminate_dirichlet": (_i32, [_p, _p]),
    "xsb_pattern_hash": (_i32, [_p, C.POINTER(_u64)]),
    "xsb_pattern_equal": (_i32, [_p, _p, C.POINTER(_i32)]),
    "xsb_add": (_i32, [_p, _p, _i32, C.POINTER(_p)]),
    "xsb_matmul": (_i32, [_p, _p, C.POINTER(_p)]),
    "xsb_dropzeros": (_i32, [_p, C.POINTER(_i64), C.POINTER(_i32)]),
    "xsb_pointblock": (_i32, [_p, _i32, C.POINTER(_p)]),
    "xsb_block_size": (_i32, [_p, C.POINTER(_i32)]),
    "xsb_fetch_blocks": (_i32, [_p, _p]),
    "xsb_emit_fdrand": (_i32, [_p, _i32, _i64, _i64, _i64, _u64, _i32, _i32]),
    "xsb_emit_fdrand_range": (_i32, [_p, _i32, _i64, _i64, _i64, _u64, _i32, _i32, _i64, _i64]),
    "xsb_emit_p1fem": (_i32, [_p, _i32, _i64, _i64, _i64, _i32]),
    "xsb_emit_p1fem_range": (_i32, [_p, _i32, _i64, _i64, _i64, _i32, _i64, _i64]),
    "xsb_emit_blockrd": (_i32, [_p, _i32, _i64, _i64, _i64, _i32, _u64, _i32]),
    "xsb_stream_count_fdrand": (_i32, [_i64, _i64, _i64, C.POINTER(_i64)]),
    "xsb_stream_count_p1fem": (_i32, [_i64, _i64, _i64, C.POINTER(_i64)]),
    "xsb_stream_count_blockrd": (_i32, [_i64, _i64, _i64, _i32, C.POINTER(_i64)]),
    "xsb_debug_fetch_staged": (_i32, [_p, _i32, _p, _p, _p, _p, _i64, C.POINTER(_i64)]),
    "xsb_synchronize": (_i32, [_p]),
    "xsb_get_stream": (_i32, [_p, C.POINTER(_p)]),
    "xsb_timer_start": (_i32, [_p]),
    "xsb_timer_stop": (_i32, [_p, C.POINTER(C.c_float)]),
    "xsb_set_profiling": (_i32, [_p, _i32]),
    "xsb_set_strategy": (_i32, [_p, _i32]),
    "xsb_mul": (_i32, [_p, _p, _p]),
    "xsb_set_grouping": (_i32, [_p, _i32]),
    "xsb_set_precount": (_i32, [_p, _i32]),
    "xsb_set_preaggregation": (_i32, [_p, _i32]),
    "xsb_get_flush_stats": (_i32, [_p, C.POINTER(FlushStats)]),
    "xsb_kernel_launches": (_i32, [_p, C.POINTER(_i64)]),
}

_lib = None


def lib() -> C.CDLL:
    """Load libxsparse_b200.so (built in-tree by build.py).  Fails loudly when absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: run `python __graft_entry__.py` (or extendablesparse.jl_b200/build.py). "
                "There is no CPU fallback."
            )
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            f = getattr(L, name)  # AttributeError if the library does not export a declared symbol
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib


def ptr(x):
    """Raw address of a numpy array (host), a torch tensor (host or device) or an int."""
    if x is None:
        return None
    if isinstance(x, int):
        return x
    if isinstance(x, np.ndarray):
        if not x.flags["C_CONTIGUOUS"]:
            raise ValueError("array must be contiguous")
        return x.ctypes.data
    if hasattr(x, "data_ptr"):
        if not x.is_contiguous():
            raise ValueError("tensor must be contiguous")
        return x.data_ptr()
    raise TypeError(f"cannot take the address of {type(x)}")


_ERR = {EBOUNDS: XsbBoundsError, ESIZE: XsbSizeError, EILLEGAL: XsbIllegalError}


def check(rc: int, handle=None):
    if rc != OK:
        msg = lib().xsb_last_error(handle)
        raise _ERR.get(rc, XsbError)(rc, msg.decode() if msg else "")


def device_count() -> int:
    c = _i32(0)
    rc = lib().xsb_device_count(C.byref(c))
    return c.value if rc == OK else 0


def stream_count_fdrand(nx, ny=1, nz=1) -> int:
    c = _i64(0)
    check(lib().xsb_stream_count_fdrand(nx, ny, nz, C.byref(c)))
    return c.value


def stream_count_p1fem(nxn, nyn, nzn) -> int:
    c = _i64(0)
    check(lib().xsb_stream_count_p1fem(nxn, nyn, nzn, C.byref(c)))
    return c.value


def stream_count_blockrd(nx, ny, nz, ns=4) -> int:
    c = _i64(0)
    check(lib().xsb_stream_count_blockrd(nx, ny, nz, ns, C.byref(c)))
    return c.value


class Handle:
    """Thin object wrapper of an `xsb_matrix*`; method names follow the C entry points."""

    def __init__(self, m, n, idx_type=I64, index_base=1, n_tid=1, device=0, slab=None):
        """slab=(n_ranks, rank, col_splits): own columns [col_splits[rank], col_splits[rank+1]) of an m x n matrix."""
        self._h = None
        h = _p()
        if slab is None:
            check(lib().xsb_create(m, n, F64, idx_type, index_base, n_tid, device, C.byref(h)))
            self.n_global, self.col_begin = int(n), 0
        else:
            n_ranks, rank, splits = slab
            arr = (_i64 * (n_ranks + 1))(*[int(x) for x in splits])
            check(lib().xsb_create_slab(m, n, n_ranks, rank, arr, F64, idx_type, index_base, device, C.byref(h)))
            self.n_global, self.col_begin = int(n), int(splits[rank])
            n = int(splits[rank + 1]) - int(splits[rank])
            self.n_ranks, self.rank = n_ranks, rank
        self._h = h
        self.m, self.n = int(m), int(n)
        self.idx_type, self.index_base, self.n_tid, self.device = idx_type, index_base, n_tid, device
        self.idx_dtype = np.int64 if idx_type == I64 else np.int32

    def close(self):
        if self._h:
            lib().xsb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _c(self, rc):
        check(rc, self._h)

    def reset(self):
        self._c(lib().xsb_reset(self._h))

    def set_csc(self, colptr, rowval, nzval):
        self._c(lib().xsb_set_csc(self._h, ptr(colptr), ptr(rowval), ptr(nzval)))

    def route_count(self):
        """Staged records per owning rank (own rank: the ones that stay)."""
        counts = (_i64 * max(self.n_ranks, 1))()
        self._c(lib().xsb_route_count(self._h, counts))
        return [int(c) for c in counts]

    def route_prepare(self, send_records, capacity):
        """Copies the records other ranks own into send_records (dest after dest); returns counts."""
        counts = (_i64 * max(self.n_ranks, 1))()
        self._c(lib().xsb_route_prepare(self._h, ptr(send_records), capacity, counts))
        return [int(c) for c in counts]

    def route_finish(self, src_rank, recv_records, count):
        self._c(lib().xsb_route_finish(self._h, int(src_rank), ptr(recv_records), count))

    def route_pack(self, send_records, caps, capacity):
        """Fixed-capacity exchange: blocks (header + caps[d] slots) for every destination d != own rank."""
        arr = (_i64 * max(self.n_ranks, 1))(*[int(c) for c in caps])
        self._c(lib().xsb_route_pack(self._h, ptr(send_records), arr, int(capacity)))

    def route_unpack(self, recv_records, caps):
        """Fixed-capacity exchange: the received blocks (sources ascending, own rank left out) become staged regions."""
        arr = (_i64 * max(self.n_ranks, 1))(*[int(c) for c in caps])
        self._c(lib().xsb_route_unpack(self._h, ptr(recv_records), arr))

    # peer exchange (NVLink peer memory; see include/xsparse_b200.h)
    def peer_exchange_create(self, caps) -> bytes:
        """caps[dst][src] (or flat, dst-major) = slots of the block src -> dst; returns this rank's 64-byte IPC handle."""
        flat = [int(c) for row in caps for c in (row if hasattr(row, "__len__") else [row])]
        assert len(flat) == self.n_ranks ** 2, "caps must be n_ranks x n_ranks"
        arr = (_i64 * len(flat))(*flat)
        out = C.create_string_buffer(64)
        self._c(lib().xsb_peer_exchange_create(self._h, arr, C.cast(out, _p)))
        return out.raw

    def peer_exchange_connect(self, handles: bytes):
        assert len(handles) == 64 * self.n_ranks
        buf = C.create_string_buffer(bytes(handles), len(handles))
        self._c(lib().xsb_peer_exchange_connect(self._h, C.cast(buf, _p)))

    def peer_exchange_connect_local(self, peers):
        arr = (_p * self.n_ranks)(*[(p._h if p is not None else None) for p in peers])
        self._c(lib().xsb_peer_exchange_connect_local(self._h, arr))

    def peer_exchange_disconnect(self):
        self._c(lib().xsb_peer_exchange_disconnect(self._h))

    def peer_exchange_destroy(self):
        self._c(lib().xsb_peer_exchange_destroy(self._h))

    def route_pack_peer(self):
        self._c(lib().xsb_route_pack_peer(self._h))

    def route_unpack_peer(self):
        self._c(lib().xsb_route_unpack_peer(self._h))

    def get_stream(self) -> int:
        """cudaStream_t of the handle (an integer address; wrap with torch.cuda.ExternalStream)."""
        v = _p()
        self._c(lib().xsb_get_stream(self._h, C.byref(v)))
        return int(v.value or 0)

    def shrink_to_fit(self):
        self._c(lib().xsb_shrink_to_fit(self._h))

    @property
    def nnz(self) -> int:
        c = _i64(0)
        self._c(lib().xsb_nnz(self._h, C.byref(c)))
        return c.value

    @property
    def pending(self) -> int:
        c = _i64(0)
        self._c(lib().xsb_pending(self._h, C.byref(c)))
        return c.value

    def reserve(self, tid, count):
        self._c(lib().xsb_reserve(self._h, tid, count))

    def insert_batch(self, I, J, V, flavour=UPDATE, tid=0, count=None):
        if count is None:
            count = len(V)
        self._c(lib().xsb_insert_batch(self._h, tid, ptr(I), ptr(J), ptr(V), count, flavour))

    def insert_triplets(self, T, flavour=UPDATE, tid=0, count=None):
        """T: `count` 16-byte triplets {u32 row, u32 col, f64 val} (numpy array of TRIPLET_DTYPE, or any
        16-byte-aligned buffer / torch tensor holding them); indices carry the handle's index base."""
        if count is None:
            count = len(T)
        self._c(lib().xsb_insert_triplets(self._h, tid, ptr(T), count, flavour))

    def _dof_array(self, dofs, name):
        if hasattr(dofs, "data_ptr"):
            want = "torch.int64" if self.idx_type == I64 else "torch.int32"
            if str(dofs.dtype) != want:
                raise TypeError(f"{name} must be {want}")
        else:
            dofs = np.ascontiguousarray(dofs, self.idx_dtype)
        if dofs.ndim != 2:
            raise ValueError(f"{name} must have shape (ncells, k)")
        return dofs

    def _element_arrays(self, dofs, Aloc=None, col_dofs=None):
        """(ncells, k) connectivity in the handle's index type and (ncells, k, k) Float64 element matrices, both
        C-contiguous: the column-major k x ncells / k x k x ncells arrays of the C ABI (Aloc[c, jl, il] is entry
        (il, jl) of element c).  With col_dofs, dofs is the (ncells, kr) row connectivity, col_dofs the (ncells, kc)
        column connectivity and Aloc has shape (ncells, kc, kr).  numpy arrays are converted, torch tensors (host or
        device) must already match.  Returns (dofs, col_dofs, Aloc, ncells, kr, kc)."""
        dofs = self._dof_array(dofs, "dofs")
        ncells, kr = (int(x) for x in dofs.shape)
        kc = kr
        if col_dofs is not None:
            col_dofs = self._dof_array(col_dofs, "col_dofs")
            if int(col_dofs.shape[0]) != ncells:
                raise ValueError(f"col_dofs must have {ncells} rows, one per element, not {int(col_dofs.shape[0])}")
            kc = int(col_dofs.shape[1])
        if Aloc is not None:
            if hasattr(Aloc, "data_ptr"):
                if str(Aloc.dtype) != "torch.float64":
                    raise TypeError("Aloc must be torch.float64")
            else:
                Aloc = np.ascontiguousarray(Aloc, np.float64)
            if tuple(Aloc.shape) != (ncells, kc, kr):
                what = "(ncells, k, k)" if col_dofs is None else "(ncells, kc, kr)"
                raise ValueError(f"Aloc must have shape {what} = {(ncells, kc, kr)}, not {tuple(Aloc.shape)}")
        return dofs, col_dofs, Aloc, ncells, kr, kc

    def insert_elements(self, dofs, Aloc, flavour=RAW, tid=0, col_dofs=None):
        """k*k*ncells calls of an element loop: call k*k*c + k*jl + il is (dofs[c, il], dofs[c, jl], Aloc[c, jl, il]).
        With col_dofs (rows and columns from different connectivities, kr and kc dofs per element): call
        kr*kc*c + kr*jl + il is (dofs[c, il], col_dofs[c, jl], Aloc[c, jl, il])."""
        dofs, col_dofs, Aloc, ncells, kr, kc = self._element_arrays(dofs, Aloc, col_dofs)
        if col_dofs is None:
            self._c(lib().xsb_insert_elements(self._h, tid, kr, ncells, ptr(dofs), ptr(Aloc), flavour))
        else:
            self._c(lib().xsb_insert_elements_rect(self._h, tid, kr, kc, ncells, ptr(dofs), ptr(col_dofs), ptr(Aloc),
                                                   flavour))

    def freeze_elements(self, dofs, col_dofs=None):
        """freeze_pattern for the stream insert_elements(dofs, ., col_dofs=col_dofs) stages; reassemble_values(Aloc)
        then takes the element matrices as they are."""
        dofs, col_dofs, _, ncells, kr, kc = self._element_arrays(dofs, None, col_dofs)
        if col_dofs is None:
            self._c(lib().xsb_freeze_elements(self._h, kr, ncells, ptr(dofs)))
        else:
            self._c(lib().xsb_freeze_elements_rect(self._h, kr, kc, ncells, ptr(dofs), ptr(col_dofs)))

    def flush(self, mode=DETERMINISTIC, combine=COMBINE_SEED):
        nnz, changed = _i64(0), _i32(0)
        self._c(lib().xsb_flush_ex(self._h, mode, combine, C.byref(nnz), C.byref(changed)))
        return nnz.value, bool(changed.value)

    def fetch_csc(self, colptr=None, rowval=None, nzval=None):
        self._c(lib().xsb_fetch_csc(self._h, ptr(colptr), ptr(rowval), ptr(nzval)))

    def fetch_csc_numpy(self):
        nnz = self.nnz
        cp = np.empty(self.n + 1, self.idx_dtype)
        rv = np.empty(nnz, self.idx_dtype)
        nz = np.empty(nnz, np.float64)
        self.fetch_csc(cp, rv if nnz else None, nz if nnz else None)
        return cp, rv, nz

    def get_values(self, I, J, out=None):
        I = np.ascontiguousarray(I, self.idx_dtype) if not hasattr(I, "data_ptr") else I
        J = np.ascontiguousarray(J, self.idx_dtype) if not hasattr(J, "data_ptr") else J
        count = len(I)
        if out is None:
            out = np.empty(count, np.float64)
        self._c(lib().xsb_get_values(self._h, ptr(I), ptr(J), ptr(out), count))
        return out

    def zero_values(self):
        self._c(lib().xsb_zero_values(self._h))

    def freeze_pattern(self, I, J, count=None):
        if count is None:
            count = len(I)
        self._c(lib().xsb_freeze_pattern(self._h, ptr(I), ptr(J), count))

    def reassemble_values(self, V, mode=DETERMINISTIC, count=None, zero_first=False):
        """zero_first: nonzeros(A) .= 0 and the re-assembly in one pass (xsb_reassemble_values_zeroed)."""
        if count is None:
            count = len(V)
        f = lib().xsb_reassemble_values_zeroed if zero_first else lib().xsb_reassemble_values
        self._c(f(self._h, ptr(V), count, mode))

    def unfreeze(self):
        self._c(lib().xsb_unfreeze(self._h))

    # a stream of GLOBAL positions frozen across column slabs (see include/xsparse_b200.h, xsb_freeze_slab)
    def _rank_counts(self):
        return (_i64 * max(getattr(self, "n_ranks", 1), 1))()

    def freeze_slab(self, I, J, count=None):
        """First step of the slab freeze: returns the positions per owning rank (own rank: the ones kept)."""
        I = np.ascontiguousarray(I, self.idx_dtype) if not hasattr(I, "data_ptr") else I
        J = np.ascontiguousarray(J, self.idx_dtype) if not hasattr(J, "data_ptr") else J
        if count is None:
            count = len(I)
        counts = self._rank_counts()
        self._c(lib().xsb_freeze_slab(self._h, ptr(I), ptr(J), count, counts))
        return [int(c) for c in counts]

    def freeze_slab_elements(self, dofs, col_dofs=None):
        """freeze_slab for the stream insert_elements(dofs, ., col_dofs=col_dofs) stages ((ncells, k) connectivity,
        or (ncells, kr) rows and (ncells, kc) columns)."""
        dofs, col_dofs, _, ncells, kr, kc = self._element_arrays(dofs, None, col_dofs)
        counts = self._rank_counts()
        if col_dofs is None:
            self._c(lib().xsb_freeze_slab_elements(self._h, kr, ncells, ptr(dofs), counts))
        else:
            self._c(lib().xsb_freeze_slab_elements_rect(self._h, kr, kc, ncells, ptr(dofs), ptr(col_dofs), counts))
        return [int(c) for c in counts]

    def freeze_slab_prepare(self, send_positions, capacity):
        """The foreign positions (8 bytes each: u32 row, u32 owner-relative column), destination after destination,
        into device memory."""
        self._c(lib().xsb_freeze_slab_prepare(self._h, ptr(send_positions), int(capacity)))

    def freeze_slab_finish(self, recv_positions, recv_counts):
        """The received positions, sources ascending (own rank left out); completes the freeze."""
        arr = self._rank_counts()
        for r, c in enumerate(recv_counts):
            arr[r] = int(c)
        self._c(lib().xsb_freeze_slab_finish(self._h, ptr(recv_positions), arr))

    def frozen_slab_counts(self):
        """(send_counts, recv_counts) of the per-step exchange of a frozen slab stream."""
        s, r = self._rank_counts(), self._rank_counts()
        self._c(lib().xsb_frozen_slab_counts(self._h, s, r))
        return [int(c) for c in s], [int(c) for c in r]

    def reassemble_slab_pack(self, V, send_values, count=None):
        """The values of the foreign positions into send_values (device float64), laid out as at prepare."""
        if isinstance(V, np.ndarray):
            V = np.ascontiguousarray(V, np.float64)
        if count is None:
            count = len(V)
        self._c(lib().xsb_reassemble_slab_pack(self._h, ptr(V), count, ptr(send_values)))

    def reassemble_slab_values(self, V, recv_values, mode=DETERMINISTIC, zero_first=False, count=None):
        """Own values V (one per position of the frozen stream) and the received ones folded into the slab."""
        if isinstance(V, np.ndarray):
            V = np.ascontiguousarray(V, np.float64)
        if isinstance(recv_values, np.ndarray):
            recv_values = np.ascontiguousarray(recv_values, np.float64)
        if count is None:
            count = len(V)
        self._c(lib().xsb_reassemble_slab_values(self._h, ptr(V), count, ptr(recv_values), int(mode),
                                                 int(bool(zero_first))))

    def mark_dirichlet(self, penalty=1.0e20):
        mk = np.zeros(self.n, np.uint8)
        self._c(lib().xsb_mark_dirichlet(self._h, penalty, ptr(mk)))
        return mk

    def eliminate_dirichlet(self, marker):
        mk = np.ascontiguousarray(marker, np.uint8) if not hasattr(marker, "data_ptr") else marker
        self._c(lib().xsb_eliminate_dirichlet(self._h, ptr(mk)))

    def mul(self, x, y=None):
        """y = A*x on the resident CSC (numpy arrays or torch tensors, host or device)."""
        if y is None:
            y = np.empty(self.m, np.float64)
        if isinstance(x, np.ndarray):
            x = np.ascontiguousarray(x, np.float64)
        self._c(lib().xsb_mul(self._h, ptr(x), ptr(y)))
        return y

    def pointblock(self, blocksize) -> "Handle":
        """pointblock(A, blocksize) (extendable.jl:292-318): a new handle holding the block matrix."""
        out = _p()
        self._c(lib().xsb_pointblock(self._h, int(blocksize), C.byref(out)))
        nb = self.n // int(blocksize)
        hb = Handle.__new__(Handle)
        hb._h = out
        hb.m = hb.n = hb.n_global = nb
        hb.col_begin = 0
        hb.idx_type, hb.index_base, hb.n_tid, hb.device = self.idx_type, self.index_base, 1, self.device
        hb.idx_dtype = self.idx_dtype
        hb.block_size = int(blocksize)
        return hb

    def fetch_blocks_numpy(self):
        """Blocks of a pointblock result: array [nnz, bs, bs] with blocks[k, jj, ii] = block k's [ii, jj]
        (every block column-major, as SMatrix stores it), in CSC order."""
        bs = _i32(0)
        self._c(lib().xsb_block_size(self._h, C.byref(bs)))
        out = np.zeros((self.nnz, bs.value, bs.value), np.float64)
        self._c(lib().xsb_fetch_blocks(self._h, ptr(out)))
        return out

    def pattern_hash(self) -> int:
        v = _u64(0)
        self._c(lib().xsb_pattern_hash(self._h, C.byref(v)))
        return v.value

    def pattern_equal(self, other: "Handle") -> bool:
        """pattern_equal(a, b) (sparsematrixcsc.jl:77-85): same colptr and rowval, compared on the device."""
        v = _i32(0)
        self._c(lib().xsb_pattern_equal(self._h, other._h, C.byref(v)))
        return bool(v.value)

    def add(self, other: "Handle", op=OP_ADD) -> "Handle":
        """A + B (op=OP_ADD) or A - B (op=OP_SUB) of two flushed matrices: SparseArrays' map(+/-, A, B) on the
        device, entries equal to zero not stored.  Returns a new plain handle, a full assembly target."""
        out = _p()
        self._c(lib().xsb_add(self._h, other._h, int(op), C.byref(out)))
        hc = Handle.__new__(Handle)
        hc._h = out
        hc.m, hc.n, hc.n_global, hc.col_begin = self.m, self.n, self.n, 0
        hc.idx_type, hc.index_base, hc.n_tid, hc.device = self.idx_type, self.index_base, 1, self.device
        hc.idx_dtype = self.idx_dtype
        return hc

    def matmul(self, other: "Handle") -> "Handle":
        """A * B of two flushed matrices: SparseArrays' spmatmul on the device (structural pattern, each entry the
        left fold in ascending k of the products).  Returns a new plain self.m x other.n handle, a full assembly
        target."""
        out = _p()
        self._c(lib().xsb_matmul(self._h, other._h, C.byref(out)))
        hc = Handle.__new__(Handle)
        hc._h = out
        hc.m, hc.n, hc.n_global, hc.col_begin = self.m, other.n, other.n, 0
        hc.idx_type, hc.index_base, hc.n_tid, hc.device = self.idx_type, self.index_base, 1, self.device
        hc.idx_dtype = self.idx_dtype
        return hc

    def dropzeros(self):
        """dropzeros!(A) in place on the device: (nnz, pattern changed)."""
        nnz, changed = _i64(0), _i32(0)
        self._c(lib().xsb_dropzeros(self._h, C.byref(nnz), C.byref(changed)))
        return nnz.value, bool(changed.value)

    def emit_fdrand(self, nx, ny=1, nz=1, seed=20240717, ones=False, flavour=UPDATE, tid=0, l_range=None):
        if l_range is None:
            self._c(lib().xsb_emit_fdrand(self._h, tid, nx, ny, nz, seed, int(bool(ones)), flavour))
        else:
            self._c(lib().xsb_emit_fdrand_range(self._h, tid, nx, ny, nz, seed, int(bool(ones)), flavour,
                                                l_range[0], l_range[1]))

    def emit_p1fem(self, nxn, nyn, nzn, flavour=RAW, tid=0, cz_range=None):
        if cz_range is None:
            self._c(lib().xsb_emit_p1fem(self._h, tid, nxn, nyn, nzn, flavour))
        else:
            self._c(lib().xsb_emit_p1fem_range(self._h, tid, nxn, nyn, nzn, flavour, cz_range[0], cz_range[1]))

    def emit_blockrd(self, nx, ny, nz, ns=4, seed=20240717, flavour=UPDATE, tid=0):
        self._c(lib().xsb_emit_blockrd(self._h, tid, nx, ny, nz, ns, seed, flavour))

    def debug_fetch_staged(self, tid=0):
        c = _i64(0)
        self._c(lib().xsb_debug_fetch_staged(self._h, tid, None, None, None, None, 0, C.byref(c)))
        n = c.value
        I = np.empty(n, self.idx_dtype)
        J = np.empty(n, self.idx_dtype)
        V = np.empty(n, np.float64)
        F = np.empty(n, np.int32)
        if n:
            self._c(lib().xsb_debug_fetch_staged(self._h, tid, ptr(I), ptr(J), ptr(V), ptr(F), n, C.byref(c)))
        return I, J, V, F

    def synchronize(self):
        self._c(lib().xsb_synchronize(self._h))

    @property
    def stream(self) -> int:
        s = _p()
        self._c(lib().xsb_get_stream(self._h, C.byref(s)))
        return s.value or 0

    def timer_start(self):
        self._c(lib().xsb_timer_start(self._h))

    def timer_stop(self) -> float:
        ms = C.c_float(0)
        self._c(lib().xsb_timer_stop(self._h, C.byref(ms)))
        return ms.value

    def set_grouping(self, grouping):
        """GROUPING_AUTO (two-pass grouping by column when the stream has column locality), GROUPING_OFF
        (always the radix sort) or GROUPING_ON (always try)."""
        self._c(lib().xsb_set_grouping(self._h, int(grouping)))

    def set_precount(self, on=True):
        """Grouping at insertion (default on): pack / emit kernels bring every chunk into column order and publish its runs."""
        self._c(lib().xsb_set_precount(self._h, 1 if on else 0))

    def set_preaggregation(self, on=True):
        self._c(lib().xsb_set_preaggregation(self._h, 1 if on else 0))

    def set_strategy(self, strategy):
        """STRATEGY_AUTO (records grouped by column, duplicates folded per column) or STRATEGY_FULLSORT ((col,row) sort)."""
        self._c(lib().xsb_set_strategy(self._h, int(strategy)))

    def set_profiling(self, on=True):
        self._c(lib().xsb_set_profiling(self._h, int(bool(on))))

    def flush_stats(self) -> dict:
        st = FlushStats()
        self._c(lib().xsb_get_flush_stats(self._h, C.byref(st)))
        return st.as_dict()

    @property
    def kernel_launches(self) -> int:
        c = _i64(0)
        self._c(lib().xsb_kernel_launches(self._h, C.byref(c)))
        return c.value
