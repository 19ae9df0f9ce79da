"""GPU parity tests: the sm_100a kernels, called through the C ABI (libdj_b200.so via ctypes),
against the CPU oracle on the same seeded inputs.  Integer work -> bit-exact."""
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _t(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _n(t):
    return t.cpu().numpy()


def test_partition_ids_match_oracle_and_golden(dj, oracle):
    kat = json.load(open(os.path.join(GOLD, "murmur3_kat.json")))
    for seed, table in kat["partition_assumed"].items():
        keys = np.array([int(k) for k in table], dtype=np.int64)
        for nparts, name in ((8, "p8"), (32, "p32"), (7, "p7")):
            want = np.array([v[name] for v in table.values()], dtype=np.int32)
            assert (_n(dj.partition_ids(_t(keys), int(seed), nparts)) == want).all()
    rng = np.random.default_rng(11)
    keys = rng.integers(-(1 << 63), (1 << 63) - 1, 300_000, dtype=np.int64)
    for nparts, hid in ((8, dj.HASH_MURMUR3), (5, dj.HASH_MURMUR3), (4, dj.HASH_IDENTITY)):
        got = _n(dj.partition_ids(_t(keys), 12345678, nparts, hid))
        assert (got == oracle.partition_ids(keys, 12345678, nparts, hid)).all()


@pytest.mark.parametrize("n,nparts,npay", [(0, 8, 1), (1, 8, 1), (4095, 8, 1), (4097, 2, 1), (250_000, 8, 1),
                                           (250_000, 32, 1), (100_003, 7, 2), (100_003, 64, 3),
                                           (1_000_000, 1024, 1), (3_000_000, 8, 1)])
def test_hash_partition_matches_oracle(dj, oracle, n, nparts, npay):
    """cudf::hash_partition contract: offsets bit-identical, each partition equal as a multiset."""
    rng = np.random.default_rng(n + nparts)
    keys = rng.integers(-(1 << 62), 1 << 62, n, dtype=np.int64)
    pays = [np.arange(n, dtype=np.int64) * (c + 1) + c for c in range(npay)]
    ko, pos, off = dj.hash_partition(_t(keys), [_t(p) for p in pays], nparts, dj.SEED_NVLINK)
    ko, pos, off = _n(ko), [_n(p) for p in pos], _n(off)
    ok, op, ooff = oracle.hash_partition(keys, pays[0], nparts, oracle.SEED_NVLINK)
    assert (off == ooff).all()
    ids = oracle.partition_ids(ko, oracle.SEED_NVLINK, nparts) if n else np.empty(0, np.int32)
    for p in range(nparts):
        assert (ids[off[p]:off[p + 1]] == p).all()
        a = np.sort(pos[0][off[p]:off[p + 1]])
        b = np.sort(op[ooff[p]:ooff[p + 1]])
        assert (a == b).all()
    # rows stay intact: payload c is a function of payload 0, key is keys[payload0]
    assert (ko == keys[pos[0]]).all() if n else True
    for c in range(1, npay):
        assert (pos[c] == pos[0] * (c + 1) + c).all()


def test_hash_partition_identity_hash_colocation(dj):
    """G4 (test/test_shuffle_on.cpp:78-83): identity hash -> all keys of a partition congruent."""
    rng = np.random.default_rng(12)
    keys = rng.integers(0, 10_000_000, 1_000_000, dtype=np.int64)
    ko, _, off = dj.hash_partition(_t(keys), [_t(keys)], 8, 0, dj.HASH_IDENTITY)
    ko, off = _n(ko), _n(off)
    for p in range(8):
        part = ko[off[p]:off[p + 1]]
        assert part.size == 0 or (part % 8 == part[0] % 8).all()


@pytest.mark.parametrize("case", json.load(open(os.path.join(GOLD, "analytical.json")))["cases"][:4])
def test_analytical_join(dj, case):
    """G1 (test/compare_against_analytical.cu:44-54,152): 3i JOIN 5j -> size/5 rows + row predicate."""
    import torch

    size = case["size"]
    i = torch.arange(size, dtype=torch.int64, device="cuda")
    (c0, c1, c2, c3), n = dj.inner_join(3 * i, i.clone(), 5 * i, i.clone())
    assert n == case["rows"]
    assert bool((c0 % 15 == 0).all()) and bool((c1 == c0 // 3).all()) and bool((c2 % 15 == 0).all())
    assert bool((c3 == c2 // 5).all()) and bool((c0 == c2).all())


@pytest.mark.parametrize("nb,np_,sel,unique", [(1000, 1000, 0.3, True), (100_000, 250_000, 0.3, True),
                                              (1_000_000, 1_000_000, 0.3, True), (1_000_000, 5_000_000, 1.0, True),
                                              (300_000, 1_200_000, 0.9, False), (5_000_000, 5_000_000, 0.3, True)])
def test_inner_join_matches_oracle(dj, oracle, nb, np_, sel, unique):
    """G3/G5: same generated tables on GPU and CPU; join equal as a row multiset, cardinality bit-identical."""
    g_o = oracle.gen_params(nb, np_, sel, 2 * max(nb, np_), unique)
    g_d = dj.gen_params(nb, np_, sel, 2 * max(nb, np_), unique)
    bk, bp = dj.generate_rows(g_d, 0, 0, 0, nb)
    pk, pp = dj.generate_rows(g_d, 1, 0, 0, np_)
    obk, obp, _ = oracle.generate_rows(g_o, 0, 0, 0, nb)
    opk, opp, hits = oracle.generate_rows(g_o, 1, 0, 0, np_)
    assert (_n(bk) == obk).all() and (_n(bp) == obp).all()  # generator parity, bit-exact
    assert (_n(pk) == opk).all() and (_n(pp) == opp).all()
    cols, n = dj.inner_join(bk, bp, pk, pp)
    n_ref, ref = oracle.inner_join(obk, obp, opk, opp)
    assert n == n_ref
    if unique:
        assert n == hits
    assert dj.multiset_checksum4(*cols) == oracle.multiset_checksum4(*ref)
    if n <= 2_000_000:
        for a, b in zip(oracle.sort_rows(*[_n(c) for c in cols]), oracle.sort_rows(*ref)):
            assert (a == b).all()


def test_inner_join_edge_cases(dj, oracle):
    import torch

    e = torch.empty(0, dtype=torch.int64, device="cuda")
    one = torch.tensor([7], dtype=torch.int64, device="cuda")
    assert dj.inner_join(e, e, one, one)[1] == 0 and dj.inner_join(one, one, e, e)[1] == 0
    assert dj.inner_join(one, one, one, one + 1)[1] == 1
    # heavy duplicates on both sides: one hot key, 3000 x 2000 pairs + bucket overflow chunks
    rng = np.random.default_rng(13)
    bk = np.concatenate([np.full(3000, 42, np.int64), rng.integers(0, 50_000, 20_000, dtype=np.int64)])
    pk = np.concatenate([np.full(2000, 42, np.int64), rng.integers(0, 50_000, 30_000, dtype=np.int64)])
    bp, pp = np.arange(bk.size, dtype=np.int64), np.arange(pk.size, dtype=np.int64) + 10**6
    cols, n = dj.inner_join(_t(bk), _t(bp), _t(pk), _t(pp), capacity=1000)  # forces the overflow retry
    n_ref, ref = oracle.inner_join(bk, bp, pk, pp)
    assert n == n_ref >= 6_000_000
    assert dj.multiset_checksum4(*cols) == oracle.multiset_checksum4(*ref)
    # extreme key values are ordinary keys (no reserved "empty" sentinel)
    ext = np.array([0, -1, np.iinfo(np.int64).min, np.iinfo(np.int64).max, 0, -1], dtype=np.int64)
    cols, n = dj.inner_join(_t(ext), _t(np.arange(6, dtype=np.int64)), _t(ext), _t(np.arange(6, dtype=np.int64)))
    assert n == oracle.inner_join(ext, np.arange(6), ext, np.arange(6))[0] == 10


def test_single_rank_distributed_join_and_host_entry(dj, oracle):
    """N=1 path of distributed_inner_join (src/distributed_join.cpp:186-199) + host-buffer entry."""
    import torch

    g_d = dj.gen_params(400_000, 600_000, 0.3, 1_200_000, True)
    g_o = oracle.gen_params(400_000, 600_000, 0.3, 1_200_000, True)
    (bk, bp), (pk, pp) = dj.generate_tables_distributed(g_d, 0, 1)
    (obk, obp), (opk, opp) = oracle.generate_tables_distributed(g_o, 0, 1)
    n_ref, ref = oracle.inner_join(obk, obp, opk, opp)
    res = dj.distributed_inner_join(None, bk, bp, pk, pp)
    assert res.n_out == n_ref and dj.multiset_checksum4(*res.cols) == oracle.multiset_checksum4(*ref)
    # left/right swapped: probe side smaller than build side -> output still left ++ right
    res2 = dj.distributed_inner_join(None, pk, pp, bk, bp)
    assert res2.n_out == n_ref
    assert dj.multiset_checksum4(res2.cols[2], res2.cols[3], res2.cols[0], res2.cols[1]) == \
        oracle.multiset_checksum4(*ref)
    # host entry
    h_in = [t.cpu().pin_memory() for t in (bk, bp, pk, pp)]
    h_out = [torch.empty(700_000, dtype=torch.int64).pin_memory() for _ in range(4)]
    n, _ = dj.distributed_inner_join_host(None, *h_in, h_out)
    assert n == n_ref
    assert oracle.multiset_checksum4(*[o[:n].numpy() for o in h_out]) == oracle.multiset_checksum4(*ref)


def test_full_size_properties_100m(dj, oracle):
    """Size-independent properties at a per-GPU size of config 2 (100M x 100M): cardinality equals the
    generator's hit count (computed on the CPU without materialising), every output row has equal keys,
    and the checksum is invariant under swapping the join sides."""
    import torch

    n = 100_000_000
    g_d = dj.gen_params(n, n, 0.3, 2 * n, True)
    g_o = oracle.gen_params(n, n, 0.3, 2 * n, True)
    bk, bp = dj.generate_rows(g_d, 0, 0, 0, n)
    pk, pp = dj.generate_rows(g_d, 1, 0, 0, n)
    hits = oracle.generate_rows(g_o, 1, 0, 0, n, materialize=False)[2]
    cols, n_out = dj.inner_join(bk, bp, pk, pp, capacity=n // 2)
    assert n_out == hits
    assert bool((cols[0] == cols[2]).all())
    assert bool((bk[cols[1]] == cols[0]).all()) and bool((pk[cols[3]] == cols[2]).all())  # payload = row id
    ck = dj.multiset_checksum4(*cols)
    del cols
    torch.cuda.empty_cache()
    cols2, n2 = dj.inner_join(pk, pp, bk, bp, capacity=n // 2)
    assert n2 == hits and dj.multiset_checksum4(cols2[2], cols2[3], cols2[0], cols2[1]) == ck


def test_bench_steps_and_dump_outputs(dj, tmp_path):
    """bench.py at a small size: --steps sets how many steps are timed in the HBM-resident and the e2e window
    (the kernel launches of each scale with it, --warmup 0 included), the timed result passes parity, and
    --dump-outputs writes that result's row count."""
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    runs = {}
    for steps in (1, 3):
        out = tmp_path / f"dump{steps}"
        r = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", str(steps), "--warmup", "0",
                            "--rows", "2000000", "--no-cpu", "--dump-outputs", str(out)], cwd=root,
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        d = json.loads([line for line in r.stdout.splitlines() if line.startswith("{")][-1])
        assert d["steps"] == steps and d["e2e"]["steps"] == steps
        assert d["parity"]["rows_ok"] and d["parity"]["checksum_ok"]
        assert np.load(out / "n_out.npy")[0] == d["output_rows"] > 0
        runs[steps] = (d["gpu_launches"], d["e2e"]["gpu_launches"], {f.name: np.load(f) for f in out.iterdir()})
    assert runs[3][0] == 3 * runs[1][0] > 0
    assert runs[3][1] == 3 * runs[1][1] > 0
    for f, a in runs[1][2].items():
        assert a.dtype == np.float64 and np.array_equal(a, runs[3][2][f]), f


def test_multi_gpu_parity_under_torchrun():
    """N >= 2 ranks over NCCL (skipped on a single-GPU box): tests/test_multi_gpu.py under torchrun."""
    import socket
    import subprocess
    import sys

    import torch

    n = min(torch.cuda.device_count(), 8)
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
                        "--master-addr", "127.0.0.1", "--master-port", str(port),
                        os.path.join("tests", "test_multi_gpu.py")], cwd=root, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "all cases passed" in r.stdout
