"""Wide tables: dj_hash_partition_cols / dj_inner_join_cols (an int64 key plus 0..15 payload columns of
4 or 8 bytes per side) and the C++ mirror's distributed_inner_join on such tables.

CPU tests call the C ABI with placeholder device pointers: every case below is rejected by the host-side
argument checks before any CUDA call.  GPU tests check the kernels against the oracle and against the
existing 2-column entry points."""
import ctypes as C
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "distributed-join_b200", "bin")
DJ_ERR_ARG, DJ_ERR_WORKSPACE = 2, 3
FAKE = 0x7F0000000000  # a non-null "device pointer": never dereferenced by the rejected calls below


def _lib():
    import djb200

    return djb200.lib()


def _ptrs(*vals):
    return (C.c_void_p * max(len(vals), 1))(*vals)


def _ints(*vals):
    return (C.c_int * max(len(vals), 1))(*vals)


# ----------------------------------------------------------------------------------------------- CPU
def test_cols_workspace_queries_need_no_gpu():
    L = _lib()
    for nb, np_ in ((1000, 1000), (100_000, 250_000), (100_000_000, 100_000_000)):
        base = L.dj_inner_join_workspace_bytes(nb, np_)
        prev = 0
        for cap in (0, 1, 1000, 10**6, 10**8):
            ws = L.dj_inner_join_cols_workspace_bytes(nb, np_, cap)
            assert ws >= base + 16 * cap
            assert ws > prev
            prev = ws
    for n, nparts in ((0, 2), (4097, 7), (10**8, 1024)):
        assert L.dj_hash_partition_cols_workspace_bytes(n, nparts) >= L.dj_hash_partition_workspace_bytes(n, nparts) \
            + 16 * n


def _partition(ncols=1, widths=(8,), cols=(FAKE,), out_cols=(FAKE,), nrows=100, key=FAKE, out_key=FAKE,
               ws_bytes=None, nparts=8):
    L = _lib()
    if ws_bytes is None:
        ws_bytes = L.dj_hash_partition_cols_workspace_bytes(nrows, nparts)
    return L.dj_hash_partition_cols(key, _ptrs(*cols), _ints(*widths), ncols, nrows, nparts, 12345678, 1, out_key,
                                    _ptrs(*out_cols), FAKE, FAKE, ws_bytes, None)


def _join(bcols=(FAKE,), bw=(8,), nbc=1, pcols=(FAKE,), pw=(4,), npc=1, nb=100, np_=200, cap=300, out_b=(FAKE,),
          out_p=(FAKE,), bk=FAKE, pk=FAKE, obk=FAKE, opk=FAKE, ws_bytes=None):
    L = _lib()
    if ws_bytes is None:
        ws_bytes = L.dj_inner_join_cols_workspace_bytes(nb, np_, cap)
    return L.dj_inner_join_cols(bk, _ptrs(*bcols), _ints(*bw), nbc, nb, pk, _ptrs(*pcols), _ints(*pw), npc, np_, obk,
                                _ptrs(*out_b), opk, _ptrs(*out_p), cap, FAKE, FAKE, ws_bytes, None)


@pytest.mark.parametrize("case", ["ncols_negative", "ncols_16", "width_2", "width_16", "null_col", "null_out_col",
                                  "null_key", "null_out_key", "workspace"])
def test_partition_cols_rejects_bad_arguments(case):
    sixteen = dict(ncols=16, widths=(8,) * 16, cols=(FAKE,) * 16, out_cols=(FAKE,) * 16)
    kw = {"ncols_negative": dict(ncols=-1), "ncols_16": sixteen, "width_2": dict(widths=(2,)),
          "width_16": dict(widths=(16,)), "null_col": dict(cols=(None,)), "null_out_col": dict(out_cols=(None,)),
          "null_key": dict(key=None), "null_out_key": dict(out_key=None), "workspace": dict(ws_bytes=4096)}[case]
    rc = _partition(**kw)
    assert rc == (DJ_ERR_WORKSPACE if case == "workspace" else DJ_ERR_ARG)
    assert b"hash_partition_cols" in _lib().dj_last_error()


@pytest.mark.parametrize("case", ["ncols_negative", "ncols_16", "width_2", "null_build_col", "null_probe_col",
                                  "null_out_build_col", "null_out_probe_col", "null_key", "null_out_key",
                                  "workspace", "workspace_for_smaller_capacity"])
def test_join_cols_rejects_bad_arguments(case):
    sixteen = dict(bcols=(FAKE,) * 16, bw=(8,) * 16, nbc=16, out_b=(FAKE,) * 16)
    L = _lib()
    kw = {"ncols_negative": dict(npc=-1), "ncols_16": sixteen, "width_2": dict(pw=(2,)),
          "null_build_col": dict(bcols=(None,)), "null_probe_col": dict(pcols=(None,)),
          "null_out_build_col": dict(out_b=(None,)), "null_out_probe_col": dict(out_p=(None,)),
          "null_key": dict(pk=None), "null_out_key": dict(obk=None), "workspace": dict(ws_bytes=64),
          "workspace_for_smaller_capacity": dict(ws_bytes=L.dj_inner_join_cols_workspace_bytes(100, 200, 100))}[case]
    rc = _join(**kw)
    assert rc == (DJ_ERR_WORKSPACE if case.startswith("workspace") else DJ_ERR_ARG)
    assert b"inner_join_cols" in L.dj_last_error()


def test_null_columns_are_fine_without_rows():
    """A null column is only an error where rows are read or written: with 0 rows / capacity the checks pass
    and the call would go on to the device, so here only the argument stage is probed, by making the workspace
    the (later) failing check."""
    assert _partition(cols=(None,), out_cols=(None,), key=None, out_key=None, nrows=0, ws_bytes=0) == DJ_ERR_WORKSPACE
    assert _join(out_b=(None,), out_p=(None,), obk=None, opk=None, cap=0, ws_bytes=0) == DJ_ERR_WORKSPACE


# ----------------------------------------------------------------------------------------------- GPU
def _t(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _n(t):
    return t.cpu().numpy()


_KINDS = ("int32", "float64", "int64")


def _col_values(kind, c, rid):
    """Payload column c (>= 1) of a row with row id `rid`: int32 (wrapping), int64, or float64 whose bit
    patterns alternate between ordinary values and NaNs with varying payloads and signs."""
    rid = np.asarray(rid, dtype=np.int64)
    if kind == "int32":
        return (rid * (2 * c + 1) + c).astype(np.int32)
    if kind == "int64":
        return rid * 1_000_003 * c - c
    nan_bits = (np.int64(0x7FF0000000000000) | ((rid * c + 1) & 0x000FFFFFFFFFFFFF)) ^ ((rid & 2) << 62)
    bits = np.where(rid % 2 == 1, nan_bits, (rid.astype(np.float64) * 0.5 + c).view(np.int64))
    return bits.view(np.float64)


def _make_cols(rid, ncols):
    """ncols payload columns: column 0 is the row id itself, the others functions of it."""
    if ncols == 0:
        return [], []
    kinds = ["rid"] + [_KINDS[c % 3] for c in range(1, ncols)]
    cols = [np.asarray(rid, dtype=np.int64)] + [_col_values(kinds[c], c, rid) for c in range(1, ncols)]
    return kinds, cols


def _check_cols(kinds, out_cols, rid):
    """Every column c >= 1 equals its function of the carried row id, bit for bit."""
    for c in range(1, len(kinds)):
        got, want = _n(out_cols[c]), _col_values(kinds[c], c, rid)
        assert got.dtype == want.dtype
        assert (got.view(np.uint8) == want.view(np.uint8)).all(), (kinds[c], c)


@pytest.mark.gpu
@pytest.mark.parametrize("ncols", [0, 1, 5, 15])
@pytest.mark.parametrize("nparts", [2, 7, 64, 1024])
@pytest.mark.parametrize("n", [0, 1, 4097, 1_000_000])
def test_hash_partition_cols_matches_oracle(dj, oracle, n, nparts, ncols):
    import torch

    rng = np.random.default_rng(7 * n + nparts + ncols)
    keys = rng.integers(-(1 << 62), 1 << 62, n, dtype=np.int64)
    rid = np.arange(n, dtype=np.int64)
    kinds, cols = _make_cols(rid, ncols)
    ko, cos, off = dj.hash_partition_cols(_t(keys), [_t(c) for c in cols], nparts)
    _, _, off_i64 = dj.hash_partition(_t(keys), [torch.arange(n, dtype=torch.int64, device="cuda")], nparts)
    ok, _, ooff = oracle.hash_partition(keys, rid, nparts, oracle.SEED_NVLINK)
    ko, off = _n(ko), _n(off)
    assert (off == _n(off_i64)).all() and (off == ooff).all()
    for p in range(nparts):
        assert (np.sort(ko[off[p]:off[p + 1]]) == np.sort(ok[ooff[p]:ooff[p + 1]])).all()
    assert len(cos) == ncols
    if ncols:
        out_rid = _n(cos[0])
        assert (np.sort(out_rid) == rid).all()  # a permutation of the input rows
        assert (ko == keys[out_rid]).all()      # ... with each row intact
        _check_cols(kinds, cos, out_rid)


def _gen_tables(dj, oracle, nb, np_, sel, unique):
    g_d = dj.gen_params(nb, np_, sel, 2 * max(nb, np_), unique)
    g_o = oracle.gen_params(nb, np_, sel, 2 * max(nb, np_), unique)
    bk, bp = dj.generate_rows(g_d, 0, 0, 0, nb)
    pk, pp = dj.generate_rows(g_d, 1, 0, 0, np_)
    obk, obp, _ = oracle.generate_rows(g_o, 0, 0, 0, nb)
    opk, opp, _ = oracle.generate_rows(g_o, 1, 0, 0, np_)
    return (bk, bp, pk, pp), (obk, obp, opk, opp)


@pytest.mark.gpu
@pytest.mark.parametrize("nb,np_,sel,unique", [(1000, 1000, 0.3, True), (1_000_000, 1_000_000, 0.3, True),
                                              (5_000_000, 5_000_000, 0.3, True), (300_000, 1_200_000, 0.9, False)])
def test_inner_join_cols_matches_oracle(dj, oracle, nb, np_, sel, unique):
    (bk, bp, pk, pp), ref_in = _gen_tables(dj, oracle, nb, np_, sel, unique)
    # payload column 0 is the generator's row id; the others are functions of it
    bkinds, bcols = _make_cols(_n(bp), 6)
    pkinds, pcols = _make_cols(_n(pp), 4)
    (bko, bco, pko, pco), n = dj.inner_join_cols(bk, [bp] + [_t(c) for c in bcols[1:]], pk,
                                                 [pp] + [_t(c) for c in pcols[1:]])
    n_ref, ref = oracle.inner_join(*ref_in)
    assert n == n_ref
    assert dj.multiset_checksum4(bko, bco[0], pko, pco[0]) == oracle.multiset_checksum4(*ref)
    _check_cols(bkinds, bco, _n(bco[0]))
    _check_cols(pkinds, pco, _n(pco[0]))


@pytest.mark.gpu
def test_inner_join_cols_edge_cases(dj, oracle):
    import torch

    e = torch.empty(0, dtype=torch.int64, device="cuda")
    one = torch.tensor([7], dtype=torch.int64, device="cuda")
    f32 = torch.tensor([1.5], dtype=torch.float32, device="cuda")
    (bko, bco, pko, pco), n = dj.inner_join_cols(e, [e], one, [one, f32])
    assert n == 0 and bko.numel() == 0 and [c.numel() for c in bco + pco] == [0, 0, 0]
    assert dj.inner_join_cols(one, [f32], e, [])[1] == 0
    # 0 payload columns on one side, then on both
    (bko, bco, pko, pco), n = dj.inner_join_cols(one, [], one, [f32])
    assert n == 1 and bco == [] and _n(bko)[0] == 7 and _n(pko)[0] == 7 and _n(pco[0])[0] == 1.5
    rng = np.random.default_rng(21)
    bk = rng.integers(0, 5000, 20_000, dtype=np.int64)
    pk = rng.integers(0, 5000, 30_000, dtype=np.int64)
    (bko, bco, pko, pco), n = dj.inner_join_cols(_t(bk), [], _t(pk), [])
    n_ref, ref = oracle.inner_join(bk, bk, pk, pk)
    assert n == n_ref and bco == [] and pco == []
    assert (_n(bko) == _n(pko)).all() and (np.sort(_n(bko)) == np.sort(ref[0])).all()
    # one hot key: 3000 x 2000 pairs, and a capacity of 1000 forces the exact retry
    bk = np.concatenate([np.full(3000, 42, np.int64), rng.integers(0, 50_000, 20_000, dtype=np.int64)])
    pk = np.concatenate([np.full(2000, 42, np.int64), rng.integers(0, 50_000, 30_000, dtype=np.int64)])
    brid, prid = np.arange(bk.size, dtype=np.int64), np.arange(pk.size, dtype=np.int64) + 10**6
    bkinds, bcols = _make_cols(brid, 3)
    pkinds, pcols = _make_cols(prid, 2)
    (bko, bco, pko, pco), n = dj.inner_join_cols(_t(bk), [_t(c) for c in bcols], _t(pk), [_t(c) for c in pcols],
                                                 capacity=1000)
    n_ref, ref = oracle.inner_join(bk, brid, pk, prid)
    assert n == n_ref >= 6_000_000
    assert dj.multiset_checksum4(bko, bco[0], pko, pco[0]) == oracle.multiset_checksum4(*ref)
    _check_cols(bkinds, bco, _n(bco[0]))
    _check_cols(pkinds, pco, _n(pco[0]))
    # extreme key values are ordinary keys
    ext = np.array([0, -1, np.iinfo(np.int64).min, np.iinfo(np.int64).max, 0, -1], dtype=np.int64)
    six = np.arange(6, dtype=np.int64)
    (bko, bco, pko, pco), n = dj.inner_join_cols(_t(ext), [_t(six)], _t(ext), [_t(six + 100)])
    n_ref, ref = oracle.inner_join(ext, six, ext, six + 100)
    assert n == n_ref == 10
    assert dj.multiset_checksum4(bko, bco[0], pko, pco[0]) == oracle.multiset_checksum4(*ref)


@pytest.mark.gpu
def test_inner_join_cols_one_column_equals_inner_join(dj, oracle):
    (bk, bp, pk, pp), _ = _gen_tables(dj, oracle, 1_000_000, 2_000_000, 0.5, False)
    (bko, (bpo,), pko, (ppo,)), n = dj.inner_join_cols(bk, [bp], pk, [pp])
    cols, n_ref = dj.inner_join(bk, bp, pk, pp)
    assert n == n_ref
    assert dj.multiset_checksum4(bko, bpo, pko, ppo) == dj.multiset_checksum4(*cols)
    for a, b in zip(oracle.sort_rows(*[_n(c) for c in (bko, bpo, pko, ppo)]), oracle.sort_rows(*[_n(c) for c in cols])):
        assert (a == b).all()


# ----------------------------------------------------------------------------------------------- C++ mirror
_CASES = 2 * 2 * 2 * 2 * 3  # key types x sizes x odf x nvlink_domain_size x table shapes


def _run(nproc, exe, *args):
    if nproc == 1:
        return subprocess.run([os.path.join(BIN, exe), *args], cwd=ROOT, capture_output=True, text=True, timeout=300,
                              env=dict(os.environ, RANK="0", WORLD_SIZE="1", LOCAL_RANK="0"))
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return subprocess.run([sys.executable, "-m", "torch.distributed.run", "--no-python", "--nnodes=1",
                           f"--nproc-per-node={nproc}", "--master-addr", "127.0.0.1", "--master-port", str(port),
                           os.path.join(BIN, exe), *args], cwd=ROOT, capture_output=True, text=True, timeout=600)


@pytest.mark.gpu
def test_wide_payload_single_rank():
    """distributed_inner_join of wide tables through the C++ mirror (test/wide_payload.cu) on one rank."""
    r = _run(1, "wide_payload")
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert r.stderr.count('Test case "wide_payload" passes successfully.') == _CASES, r.stderr[-4000:]


@pytest.mark.gpu
def test_wide_payload_multi_rank():
    import torch

    n = min(torch.cuda.device_count(), 8)
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    r = _run(n, "wide_payload")
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert r.stderr.count('Test case "wide_payload" passes successfully.') == _CASES, r.stderr[-4000:]
