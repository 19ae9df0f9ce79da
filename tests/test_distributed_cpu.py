"""CPU multi-process tests (gloo, world_size 2): BASELINE config 0 through the oracle, and the
launcher contract of bench.py's reference arm."""
import json
import os
import socket
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _torchrun(nproc, script, *args, timeout=300):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()), script, *map(str, args)]
    env = dict(os.environ, OMP_NUM_THREADS="2")
    return subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=timeout)


@pytest.mark.parametrize("total,odf", [(1_000_000, 1), (200_000, 4)])
def test_config0_two_rank_gloo_pipeline(total, odf):
    r = _torchrun(2, os.path.join("tests", "dist_worker_gloo.py"), total, odf)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "DIST_OK" in r.stdout


def test_bench_reference_arm_under_torchrun_prints_one_line(monkeypatch):
    """--impl reference under torchrun: rank 0 alone runs and prints the JSON line; other ranks exit 0."""
    env_rows = {"DJ_CPU_SAMPLE_ROWS": "200000"}
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
           "127.0.0.1", "--master-port", str(_free_port()), "bench.py", "--impl", "reference", "--gpus", "2",
           "--steps", "1", "--warmup", "0"]
    r = subprocess.run(cmd, cwd=ROOT, env=dict(os.environ, **env_rows), capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["cpu_baseline"]["kind"] == "port" and d["value"] > 0
    assert d["e2e"]["h2d_bytes_per_step"] == 0


def test_bench_dump_outputs_is_independent_of_row_order(oracle, tmp_path):
    """--dump-outputs samples the joined rows by content (the probe row id) and sorts them, so two runs that return
    the same row multiset in different orders dump identical files, and every value survives float64 exactly.
    The table is larger than the sample, so the dump holds a strict subset of the joined rows.  Rows whose probe
    payload is not a probe row id (a corrupt result) are left out instead of failing the dump."""
    import numpy as np
    import torch

    import bench

    n = 3_000_000
    assert n > bench.DUMP_PROBE_ROWS
    g = oracle.gen_params(n, n, 0.3, 2 * n, True)
    bk, bp, _ = oracle.generate_rows(g, 0, 0, 0, n)
    pk, pp, hits = oracle.generate_rows(g, 1, 0, 0, n)
    n_out, cols = oracle.inner_join(bk, bp, pk, pp)
    bad = [np.array([7, 7], np.int64), np.array([1, 2], np.int64), np.array([7, 7], np.int64),
           np.array([-1, n], np.int64)]
    dumps = []
    for seed, extra in ((1, False), (2, False), (3, True)):
        perm = np.random.default_rng(seed).permutation(n_out)
        rows = [np.concatenate([c[perm], b]) if extra else c[perm] for c, b in zip(cols, bad)]
        bench.dump_outputs(str(tmp_path / str(seed)), [torch.from_numpy(c) for c in rows], n_out, n, 1, 0)
        dumps.append({f: np.load(tmp_path / str(seed) / f"{f}.npy") for f in ("n_out",) + bench.DUMP_COLS})
    for d in dumps[1:]:
        for f, a in dumps[0].items():
            assert a.dtype == np.float64 and np.array_equal(a, d[f]), f
    assert dumps[0]["n_out"][0] == n_out == hits
    ids = np.random.default_rng(bench.DUMP_SEED).choice(n, bench.DUMP_PROBE_ROWS, replace=False)
    keep = np.isin(cols[3], ids)
    assert 0 < keep.sum() < n_out
    want = oracle.sort_rows(*[c[keep] for c in cols][::-1])[::-1]  # right_payload is the primary sort key
    for f, w in zip(bench.DUMP_COLS, want):
        assert np.array_equal(dumps[0][f], w.astype(np.float64)), f


def test_bench_import_does_not_pin_openmp():
    """Regression: OMP_PROC_BIND / OMP_PLACES exported at import time pinned EVERY rank's main thread to core 0
    (libgomp binds the initial thread): 105 instead of 9.5 ms/step at N=8.  They may only be set by the
    process that runs a CPU leg, right before the oracle is loaded."""
    import subprocess
    import sys

    code = ("import os, sys; os.environ.pop('OMP_PROC_BIND', None); os.environ.pop('OMP_PLACES', None); "
            "sys.argv=['bench.py']; import bench; "
            "assert 'OMP_PROC_BIND' not in os.environ and 'OMP_PLACES' not in os.environ; "
            "bench.pin_openmp_for_cpu_arm(); assert os.environ['OMP_PROC_BIND'] == 'close'; print('ok')")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr
