"""djb200 -- ctypes binding of libdj_b200.so (include/dj_b200.h) for tests, bench.py and smoke().

PyTorch is used only as plumbing: device memory (tensors), streams and torch.distributed for
process launch / unique-id broadcast.  Every compute call goes through the C ABI into the
hand-written sm_100a kernels; there is NO CPU or PyTorch fallback -- if the shared library is
missing or a call fails this module raises.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "lib", "libdj_b200.so")

HASH_IDENTITY = 0
HASH_MURMUR3 = 1
SEED_NVLINK = 12345678  # src/distributed_join.cpp:211
SEED_IB = 87654321  # src/distributed_join.cpp:160
DEFAULT_HASH_SEED = 0
GEN_SEED = 1234  # generate_dataset/generate_dataset.cuh:44

ERR_WORKSPACE = 3
ERR_OVERFLOW = 5


class DjError(RuntimeError):
    pass


class GenParams(C.Structure):
    _fields_ = [
        ("nb", C.c_int64),
        ("np", C.c_int64),
        ("rand_max", C.c_int64),
        ("selectivity", C.c_double),
        ("seed", C.c_uint64),
        ("unique_build_keys", C.c_int32),
        ("pad", C.c_int32),
    ]


class JoinOptions(C.Structure):
    _fields_ = [
        ("over_decom_factor", C.c_int),
        ("report_timing", C.c_int),
        ("t_partition_ms", C.c_double),
        ("t_comm_ms", C.c_double),
        ("t_join_ms", C.c_double),
        ("bytes_sent", C.c_int64),
        ("workspace_needed", C.c_int64),
        ("measure_exchange", C.c_int),
        ("pad_", C.c_int),
        ("t_exchange_ms", C.c_double * 2),
        ("t_exchange_total_ms", C.c_double),
    ]


# every symbol include/dj_b200.h declares (checked by the CPU test-suite)
ABI_SYMBOLS = [
    "dj_version", "dj_last_error", "dj_kernel_launch_count", "dj_profile_enable", "dj_profile_read",
    "dj_partition_ids_i64",
    "dj_hash_partition_workspace_bytes", "dj_hash_partition_i64", "dj_inner_join_workspace_bytes",
    "dj_inner_join_i64", "dj_hash_partition_cols_workspace_bytes", "dj_hash_partition_cols",
    "dj_inner_join_cols_workspace_bytes", "dj_inner_join_cols", "dj_generate_build_bitmap", "dj_generate_rows_i64", "dj_multiset_checksum4",
    "dj_comm_unique_id", "dj_comm_create", "dj_comm_destroy", "dj_comm_release_workspace", "dj_comm_nccl_handle",
    "dj_comm_rank",
    "dj_comm_size",
    "dj_comm_allgather_i64", "dj_comm_barrier", "dj_all_to_all", "dj_comm_group_start",
    "dj_comm_group_end", "dj_comm_send", "dj_comm_recv", "dj_distributed_inner_join_workspace_bytes",
    "dj_distributed_inner_join_i64", "dj_distributed_inner_join_host_workspace_bytes",
    "dj_distributed_inner_join_i64_host",
]

_lib = None


def lib() -> C.CDLL:
    """Load libdj_b200.so; fail loudly when it has not been built (no fallback path exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DjError(f"{LIB_PATH} is missing: build it with `make -C distributed-join_b200` "
                      "(or __graft_entry__.build()); there is no CPU fallback")
    L = C.CDLL(LIB_PATH)
    vp, i64, u32, sz = C.c_void_p, C.c_int64, C.c_uint32, C.c_size_t
    L.dj_version.restype = C.c_int
    L.dj_last_error.restype = C.c_char_p
    L.dj_kernel_launch_count.restype = i64
    L.dj_profile_enable.argtypes = [C.c_int]
    L.dj_profile_read.argtypes = [C.POINTER(C.c_double), C.POINTER(i64)]
    L.dj_partition_ids_i64.argtypes = [vp, i64, u32, C.c_int, C.c_int, vp, vp]
    L.dj_hash_partition_workspace_bytes.restype = sz
    L.dj_hash_partition_workspace_bytes.argtypes = [i64, C.c_int]
    L.dj_hash_partition_i64.argtypes = [vp, C.POINTER(vp), C.c_int, i64, C.c_int, u32, C.c_int, vp,
                                        C.POINTER(vp), vp, vp, sz, vp]
    L.dj_inner_join_workspace_bytes.restype = sz
    L.dj_inner_join_workspace_bytes.argtypes = [i64, i64]
    L.dj_inner_join_i64.argtypes = [vp, vp, i64, vp, vp, i64, vp, vp, vp, vp, i64, vp, vp, sz, vp]
    pvp, pint = C.POINTER(vp), C.POINTER(C.c_int)
    L.dj_hash_partition_cols_workspace_bytes.restype = sz
    L.dj_hash_partition_cols_workspace_bytes.argtypes = [i64, C.c_int]
    L.dj_hash_partition_cols.argtypes = [vp, pvp, pint, C.c_int, i64, C.c_int, u32, C.c_int, vp, pvp, vp, vp, sz,
                                         vp]
    L.dj_inner_join_cols_workspace_bytes.restype = sz
    L.dj_inner_join_cols_workspace_bytes.argtypes = [i64, i64, i64]
    L.dj_inner_join_cols.argtypes = [vp, pvp, pint, C.c_int, i64, vp, pvp, pint, C.c_int, i64, vp, pvp, vp, pvp, i64,
                                     vp, vp, sz, vp]
    L.dj_generate_build_bitmap.argtypes = [C.POINTER(GenParams), C.c_int, vp, vp]
    L.dj_generate_rows_i64.argtypes = [C.POINTER(GenParams), C.c_int, C.c_int, i64, i64, vp, vp, vp, vp]
    L.dj_multiset_checksum4.argtypes = [vp, vp, vp, vp, i64, vp, vp]
    L.dj_comm_unique_id.argtypes = [vp]
    L.dj_comm_create.argtypes = [C.c_int, C.c_int, vp, C.POINTER(vp)]
    L.dj_comm_destroy.argtypes = [vp]
    L.dj_comm_release_workspace.argtypes = [vp]
    L.dj_comm_rank.argtypes = [vp]
    L.dj_comm_size.argtypes = [vp]
    L.dj_comm_allgather_i64.argtypes = [vp, C.POINTER(i64), C.c_int, C.POINTER(i64), vp]
    L.dj_comm_barrier.argtypes = [vp, vp]
    L.dj_all_to_all.argtypes = [vp, C.c_int, C.POINTER(C.c_int), C.c_int, C.POINTER(vp), C.POINTER(vp),
                                C.POINTER(i64), C.POINTER(i64), C.POINTER(C.c_int), C.c_int, C.c_int, vp]
    L.dj_comm_group_start.argtypes = [vp]
    L.dj_comm_group_end.argtypes = [vp]
    L.dj_comm_send.argtypes = [vp, vp, i64, C.c_int, vp]
    L.dj_comm_recv.argtypes = [vp, vp, i64, C.c_int, vp]
    L.dj_distributed_inner_join_workspace_bytes.restype = sz
    L.dj_distributed_inner_join_workspace_bytes.argtypes = [i64, i64, C.c_int, C.c_int]
    L.dj_distributed_inner_join_i64.argtypes = [vp, vp, vp, i64, vp, vp, i64, vp, vp, vp, vp, i64,
                                                C.POINTER(i64), C.POINTER(JoinOptions), vp, sz, vp]
    L.dj_distributed_inner_join_host_workspace_bytes.restype = sz
    L.dj_distributed_inner_join_host_workspace_bytes.argtypes = [i64, i64, i64, C.c_int, C.c_int]
    L.dj_distributed_inner_join_i64_host.argtypes = L.dj_distributed_inner_join_i64.argtypes
    _lib = L
    return L


def _check(rc: int, allow=()):
    if rc != 0 and rc not in allow:
        raise DjError(f"libdj_b200 error {rc}: {lib().dj_last_error().decode()}")
    return rc


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _i64dev(t: torch.Tensor) -> torch.Tensor:
    if not (t.is_cuda and t.dtype == torch.int64 and t.is_contiguous()):
        raise DjError("expected a contiguous int64 CUDA tensor")
    return t


def kernel_launch_count() -> int:
    return int(lib().dj_kernel_launch_count())


PROF_CATEGORIES = ("hist", "scatter", "join", "other")


def profile_enable(on: bool):
    _check(lib().dj_profile_enable(1 if on else 0))


def profile_read():
    """{category: (milliseconds, launches)} since the last read (device time from CUDA events)."""
    ms = (C.c_double * 4)()
    n = (C.c_int64 * 4)()
    _check(lib().dj_profile_read(ms, n))
    return {c: (ms[i], n[i]) for i, c in enumerate(PROF_CATEGORIES)}


def workspace(nbytes: int, device=None) -> torch.Tensor:
    return torch.empty(int(nbytes), dtype=torch.uint8, device=device or "cuda")


# ----------------------------------------------------------------------------- single-GPU stages
def partition_ids(keys, seed, nparts, hash_id=HASH_MURMUR3):
    keys = _i64dev(keys)
    out = torch.empty(keys.numel(), dtype=torch.int32, device=keys.device)
    _check(lib().dj_partition_ids_i64(_ptr(keys), keys.numel(), seed, hash_id, nparts, _ptr(out), _stream()))
    return out


def hash_partition(keys, payloads, nparts, seed=SEED_NVLINK, hash_id=HASH_MURMUR3):
    """cudf::hash_partition replacement.  Returns (keys_out, [payload_out...], offsets[nparts+1])."""
    keys = _i64dev(keys)
    payloads = [_i64dev(p) for p in payloads]
    n = keys.numel()
    ko = torch.empty_like(keys)
    pos = [torch.empty_like(p) for p in payloads]
    offsets = torch.empty(nparts + 1, dtype=torch.int64, device=keys.device)
    ws = workspace(lib().dj_hash_partition_workspace_bytes(n, nparts), keys.device)
    vp = C.c_void_p
    pin = (vp * len(payloads))(*[p.data_ptr() for p in payloads])
    pout = (vp * len(payloads))(*[p.data_ptr() for p in pos])
    _check(lib().dj_hash_partition_i64(_ptr(keys), pin, len(payloads), n, nparts, seed, hash_id, _ptr(ko), pout,
                                       _ptr(offsets), _ptr(ws), ws.numel(), _stream()))
    return ko, pos, offsets


def inner_join(bk, bp, pk, pp, capacity=None, ws=None):
    """cudf::inner_join replacement on device tensors.
    Returns ((build key, build payload, probe key, probe payload) trimmed to n_out, n_out)."""
    bk, bp, pk, pp = map(_i64dev, (bk, bp, pk, pp))
    nb, np_ = bk.numel(), pk.numel()
    if capacity is None:
        capacity = max(np_, 1)
    dev = bk.device
    while True:
        outs = [torch.empty(capacity, dtype=torch.int64, device=dev) for _ in range(4)]
        cnt = torch.zeros(1, dtype=torch.int64, device=dev)
        if ws is None:
            ws = workspace(lib().dj_inner_join_workspace_bytes(nb, np_), dev)
        _check(lib().dj_inner_join_i64(_ptr(bk), _ptr(bp), nb, _ptr(pk), _ptr(pp), np_, *[_ptr(o) for o in outs],
                                       capacity, _ptr(cnt), _ptr(ws), ws.numel(), _stream()))
        n = int(cnt.item())
        if n <= capacity:
            return tuple(o[:n] for o in outs), n
        capacity = n  # exact retry, as dj_b200.h documents


MAX_PAYLOAD_COLUMNS = 15  # DJ_MAX_PAYLOAD_COLUMNS


def _cols_dev(cols):
    """Payload columns of a wide table: contiguous CUDA tensors of any 4- or 8-byte dtype, moved bitwise."""
    cols = list(cols)
    for c in cols:
        if not (c.is_cuda and c.is_contiguous() and c.dim() == 1 and c.element_size() in (4, 8)):
            raise DjError("expected contiguous 1-D CUDA tensors with 4- or 8-byte elements")
    return cols


def _col_arrays(cols):
    """(host array of device pointers, host array of widths) for the _cols ABI."""
    vp = C.c_void_p
    return (vp * max(len(cols), 1))(*[c.data_ptr() for c in cols]), \
        (C.c_int * max(len(cols), 1))(*[c.element_size() for c in cols])


def hash_partition_cols(keys, cols, nparts, seed=SEED_NVLINK, hash_id=HASH_MURMUR3):
    """cudf::hash_partition of a wide table: an int64 key plus 0..15 payload columns of any 4- or 8-byte
    dtype.  Returns (keys_out, [col_out...], offsets[nparts+1]); offsets equal hash_partition's."""
    keys = _i64dev(keys)
    cols = _cols_dev(cols)
    n = keys.numel()
    ko = torch.empty_like(keys)
    cos = [torch.empty_like(c) for c in cols]
    offsets = torch.empty(nparts + 1, dtype=torch.int64, device=keys.device)
    ws = workspace(lib().dj_hash_partition_cols_workspace_bytes(n, nparts), keys.device)
    pin, widths = _col_arrays(cols)
    pout, _ = _col_arrays(cos)
    _check(lib().dj_hash_partition_cols(_ptr(keys), pin, widths, len(cols), n, nparts, seed, hash_id, _ptr(ko), pout,
                                        _ptr(offsets), _ptr(ws), ws.numel(), _stream()))
    return ko, cos, offsets


def inner_join_cols(bk, bcols, pk, pcols, capacity=None):
    """cudf::inner_join of wide tables: int64 keys plus 0..15 payload columns per side of any 4- or 8-byte
    dtype.  Returns ((build key, [build cols], probe key, [probe cols]) trimmed to n_out, n_out)."""
    bk, pk = _i64dev(bk), _i64dev(pk)
    bcols, pcols = _cols_dev(bcols), _cols_dev(pcols)
    nb, np_ = bk.numel(), pk.numel()
    if capacity is None:
        capacity = max(np_, 1)
    dev = bk.device
    bin_, bw = _col_arrays(bcols)
    pin, pw = _col_arrays(pcols)
    while True:
        bko, pko = (torch.empty(capacity, dtype=torch.int64, device=dev) for _ in range(2))
        bout = [torch.empty(capacity, dtype=c.dtype, device=dev) for c in bcols]
        pout = [torch.empty(capacity, dtype=c.dtype, device=dev) for c in pcols]
        cnt = torch.zeros(1, dtype=torch.int64, device=dev)
        ws = workspace(lib().dj_inner_join_cols_workspace_bytes(nb, np_, capacity), dev)  # grows with capacity
        _check(lib().dj_inner_join_cols(_ptr(bk), bin_, bw, len(bcols), nb, _ptr(pk), pin, pw, len(pcols), np_,
                                        _ptr(bko), _col_arrays(bout)[0], _ptr(pko), _col_arrays(pout)[0], capacity,
                                        _ptr(cnt), _ptr(ws), ws.numel(), _stream()))
        n = int(cnt.item())
        if n <= capacity:
            return (bko[:n], [c[:n] for c in bout], pko[:n], [c[:n] for c in pout]), n
        capacity = n  # exact retry, as dj_b200.h documents


def gen_params(nb, np_, selectivity, rand_max, unique=True, seed=GEN_SEED) -> GenParams:
    return GenParams(int(nb), int(np_), int(rand_max), float(selectivity), int(seed), 1 if unique else 0, 0)


def build_bitmap(g: GenParams, src: int, device="cuda") -> torch.Tensor:
    bm = torch.empty((g.rand_max + 1 + 31) // 32, dtype=torch.int32, device=device)
    _check(lib().dj_generate_build_bitmap(C.byref(g), src, _ptr(bm), _stream()))
    return bm


def generate_rows(g: GenParams, which: int, src: int, row_begin: int, count: int, bitmap=None, device="cuda",
                  out=None):
    if which == 1 and not g.unique_build_keys and bitmap is None:
        bitmap = build_bitmap(g, src, device)
    if out is None:
        keys = torch.empty(count, dtype=torch.int64, device=device)
        pay = torch.empty(count, dtype=torch.int64, device=device)
    else:
        keys, pay = out
    _check(lib().dj_generate_rows_i64(C.byref(g), which, src, row_begin, count, _ptr(bitmap), _ptr(keys), _ptr(pay),
                                      _stream()))
    return keys, pay


def generate_tables_distributed(g: GenParams, rank: int, world: int, device="cuda"):
    """generate_tables_distributed (src/generate_table.cuh:155-272) without the exchange: every
    row is a closed-form function of (source rank, row), so rank `rank` directly generates the
    rows each source would have dealt to it, in source order."""
    tables = []
    for which, n in ((0, g.nb), (1, g.np)):
        chunk = n // world
        keys = torch.empty(chunk * world, dtype=torch.int64, device=device)
        pay = torch.empty(chunk * world, dtype=torch.int64, device=device)
        for s in range(world):
            bm = build_bitmap(g, s, device) if (which == 1 and not g.unique_build_keys) else None
            generate_rows(g, which, s, chunk * rank, chunk, bm, device,
                          out=(keys[s * chunk:(s + 1) * chunk], pay[s * chunk:(s + 1) * chunk]))
        tables.append((keys, pay))
    return tables[0], tables[1]


def multiset_checksum4(c0, c1, c2, c3):
    cols = [_i64dev(c) for c in (c0, c1, c2, c3)]
    out = torch.zeros(2, dtype=torch.int64, device=cols[0].device)
    _check(lib().dj_multiset_checksum4(*[_ptr(c) for c in cols], cols[0].numel(), _ptr(out), _stream()))
    a, b = out.tolist()
    return a & 0xFFFFFFFFFFFFFFFF, b & 0xFFFFFFFFFFFFFFFF


# ----------------------------------------------------------------------------- communication
class Comm:
    """NCCL communicator owned by libdj_b200 (replaces NCCLCommunicator, src/communicator.cpp:799-875).
    The unique id is broadcast with torch.distributed when a process group exists."""

    def __init__(self, rank: int = 0, size: int = 1, unique_id: bytes | None = None):
        self.rank, self.size = rank, size
        h = C.c_void_p()
        idbuf = (C.c_char * 128).from_buffer_copy(unique_id) if unique_id is not None else None
        _check(lib().dj_comm_create(rank, size, idbuf, C.byref(h)))
        self.handle = h

    @staticmethod
    def unique_id() -> bytes:
        buf = (C.c_char * 128)()
        _check(lib().dj_comm_unique_id(buf))
        return bytes(buf)

    @classmethod
    def from_torch_distributed(cls):
        import torch.distributed as dist

        if not dist.is_initialized() or dist.get_world_size() == 1:
            return cls(0, 1, None)
        rank, size = dist.get_rank(), dist.get_world_size()
        dev = torch.device("cuda", torch.cuda.current_device())
        if rank == 0:
            idt = torch.tensor(list(cls.unique_id()), dtype=torch.uint8, device=dev)
        else:
            idt = torch.zeros(128, dtype=torch.uint8, device=dev)
        dist.broadcast(idt, 0)
        return cls(rank, size, bytes(idt.cpu().tolist()))

    def allgather_i64(self, values):
        n = len(values)
        mine = (C.c_int64 * n)(*values)
        allv = (C.c_int64 * (n * self.size))()
        _check(lib().dj_comm_allgather_i64(self.handle, mine, n, allv, _stream()))
        return list(allv)

    def barrier(self):
        _check(lib().dj_comm_barrier(self.handle, _stream()))

    def release_workspace(self):
        """Collective: close the peers' CUDA IPC mappings of join workspaces (call before freeing one)."""
        _check(lib().dj_comm_release_workspace(self.handle))

    def destroy(self):
        if self.handle:
            lib().dj_comm_destroy(self.handle)
            self.handle = None


@dataclass
class JoinResult:
    cols: tuple  # (left key, left payload, right key, right payload), trimmed
    n_out: int
    options: JoinOptions


def distributed_inner_join(comm, lk, lp, rk, rp, odf=1, capacity=None, ws=None, outs=None, report_timing=False,
                           measure_exchange=False):
    """distributed_inner_join (src/distributed_join.cpp:134-340) on device tensors through the C ABI.
    Both retry loops are collective: every rank receives DJ_ERR_OVERFLOW / DJ_ERR_WORKSPACE together."""
    lk, lp, rk, rp = map(_i64dev, (lk, lp, rk, rp))
    nl, nr = lk.numel(), rk.numel()
    world = comm.size if comm else 1
    dev = lk.device
    if capacity is None:
        capacity = max(nl, nr, 1)
    if ws is None:
        ws = workspace(lib().dj_distributed_inner_join_workspace_bytes(nl, nr, world, odf), dev)
    while True:
        if outs is None or outs[0].numel() < capacity:
            outs = [torch.empty(capacity, dtype=torch.int64, device=dev) for _ in range(4)]
        cnt = C.c_int64(0)
        opts = JoinOptions(odf, 1 if report_timing else 0)
        opts.measure_exchange = 1 if measure_exchange else 0
        rc = _check(lib().dj_distributed_inner_join_i64(comm.handle if comm else None, _ptr(lk), _ptr(lp), nl,
                                                        _ptr(rk), _ptr(rp), nr, *[_ptr(o) for o in outs], capacity,
                                                        C.byref(cnt), C.byref(opts), _ptr(ws), ws.numel(), _stream()),
                    allow=(ERR_OVERFLOW, ERR_WORKSPACE) if world > 1 else (ERR_OVERFLOW,))
        n = cnt.value
        if rc == 0:
            return JoinResult(tuple(o[:n] for o in outs), n, opts)
        if rc == ERR_WORKSPACE:
            # a rank receives more rows than the balanced estimate (skewed slices / hot keys): peers unmap
            # the old workspace, everybody grows to what the library asked for, and all retry
            comm.release_workspace()
            need = int(opts.workspace_needed)
            ws = workspace(max(ws.numel(), need + need // 8), dev)
            continue
        # every rank must retry together: agree on the largest need
        need = max(comm.allgather_i64([n])) if comm and comm.size > 1 else n
        capacity = need
        outs = None


def distributed_inner_join_host(comm, h_lk, h_lp, h_rk, h_rp, h_outs, odf=1, ws=None):
    """End-to-end entry: HOST (pinned) inputs and outputs, copies inside the call."""
    nl, nr = h_lk.numel(), h_rk.numel()
    capacity = h_outs[0].numel()
    world = comm.size if comm else 1
    if ws is None:
        ws = workspace(lib().dj_distributed_inner_join_host_workspace_bytes(nl, nr, capacity, world, odf))
    cnt = C.c_int64(0)
    opts = JoinOptions(odf, 0, 0, 0, 0, 0)
    _check(lib().dj_distributed_inner_join_i64_host(comm.handle if comm else None, _ptr(h_lk), _ptr(h_lp), nl,
                                                    _ptr(h_rk), _ptr(h_rp), nr, *[_ptr(o) for o in h_outs], capacity,
                                                    C.byref(cnt), C.byref(opts), _ptr(ws), ws.numel(), _stream()))
    return cnt.value, opts
