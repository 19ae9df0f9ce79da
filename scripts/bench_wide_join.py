"""Wide-table join on one GPU: dj_inner_join_cols (late materialization) against the key + payload join.

    python scripts/bench_wide_join.py > profiles/wide_join_b200.txt

Workload: generator tables of 400 M x 400 M rows, unique build keys, selectivity 0.3 (about 120 M output
rows); payload column 0 of each side is the generator's row id and the others are functions of it.  Far
larger than the 126 MB L2.  Variants, each on the same keys:

    baseline    dj_inner_join_i64 (key + one int64 payload per side)
    cols=1/3/7  dj_inner_join_cols with 1, 3 and 7 int64 payload columns per side
    mixed7      dj_inner_join_cols with 7 columns per side, int64 and int32 alternating

Each variant: 2 warm-up calls, then 5 calls timed one by one with CUDA events (median reported), then one
more call with dj_profile_enable for the device time per kernel category.  The join kernels (hist, scatter,
join) are the same in every variant; "other" holds the partition passes' offset scans plus, for the _cols
variants, the iota and the two gathers, so gather time = other - other(baseline).  Gather bytes are counted
algorithmically: per output row and payload column one 32-byte sector read plus the column width written,
plus one 8-byte index read per output row and side.  Outputs are preallocated at the exact row count, so no
call retries.  The 1-column result's multiset checksum must equal the baseline's."""
import ctypes as C
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "distributed-join_b200"))
import djb200 as dj  # noqa: E402

ROWS = int(os.environ.get("WIDE_JOIN_ROWS", 400_000_000))
SELECTIVITY = 0.3
WARMUP, TIMED = 2, 5


def gpu_info():
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                          str(torch.cuda.current_device())], capture_output=True, text=True)
    return smi.stdout.strip() or torch.cuda.get_device_name()


def timed(call):
    """Median of TIMED event-timed calls after WARMUP calls, then one profiled call's categories."""
    for _ in range(WARMUP):
        call()
    times = []
    for _ in range(TIMED):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        call()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    dj.profile_read()  # drop anything recorded before
    dj.profile_enable(True)
    call()
    torch.cuda.synchronize()
    prof = dj.profile_read()
    dj.profile_enable(False)
    return sorted(times)[TIMED // 2], times, prof


def payload_cols(rid, kinds):
    """Payload columns of one side: column 0 is the row id, column c a function of it of dtype kinds[c]."""
    cols = [rid]
    for c, kind in enumerate(kinds[1:], start=1):
        v = rid * (2 * c + 1) + c
        cols.append(v.to(torch.int32) if kind == "int32" else v)
    return cols


def main():
    torch.cuda.set_device(0)
    L = dj.lib()
    st = dj._stream()
    g = dj.gen_params(ROWS, ROWS, SELECTIVITY, 2 * ROWS, True)
    bk, bp = dj.generate_rows(g, 0, 0, 0, ROWS)
    pk, pp = dj.generate_rows(g, 1, 0, 0, ROWS)
    dev = bk.device
    print(f"gpu: {gpu_info()}")
    print(f"tables: {ROWS} x {ROWS} rows, unique build keys, selectivity {SELECTIVITY}; "
          f"{WARMUP} warm-up + {TIMED} timed calls per variant (median), CUDA events")
    report = {"gpu": gpu_info(), "rows": ROWS, "selectivity": SELECTIVITY, "variants": {}}

    # ---- baseline: dj_inner_join_i64
    cnt = torch.zeros(1, dtype=torch.int64, device=dev)
    ws = dj.workspace(L.dj_inner_join_workspace_bytes(ROWS, ROWS), dev)
    cap = ROWS
    outs = [torch.empty(cap, dtype=torch.int64, device=dev) for _ in range(4)]

    def base_call():
        dj._check(L.dj_inner_join_i64(dj._ptr(bk), dj._ptr(bp), ROWS, dj._ptr(pk), dj._ptr(pp), ROWS,
                                      *[dj._ptr(o) for o in outs], cap, dj._ptr(cnt), dj._ptr(ws), ws.numel(), st))

    base_call()
    n = int(cnt.item())
    assert n <= cap
    ms, times, prof = timed(base_call)
    base_sum = dj.multiset_checksum4(*[o[:n] for o in outs])
    base_other = prof["other"][0]
    print(f"baseline dj_inner_join_i64: {n} rows, {ms:.2f} ms median (calls {', '.join(f'{t:.2f}' for t in times)}); "
          + ", ".join(f"{k} {v[0]:.2f} ms/{v[1]}" for k, v in prof.items()))
    report["n_out"] = n
    report["variants"]["baseline"] = {"ms": ms, "calls_ms": times, "profile": prof}
    del outs, ws
    torch.cuda.empty_cache()

    # ---- dj_inner_join_cols variants, outputs sized exactly at n
    variants = [("cols=1", ["int64"]), ("cols=3", ["int64"] * 3), ("cols=7", ["int64"] * 7),
                ("mixed7", ["int64", "int32", "int64", "int32", "int64", "int32", "int64"])]
    for name, kinds in variants:
        bcols, pcols = payload_cols(bp, kinds), payload_cols(pp, kinds)
        bout = [torch.empty(n, dtype=c.dtype, device=dev) for c in bcols]
        pout = [torch.empty(n, dtype=c.dtype, device=dev) for c in pcols]
        bko, pko = torch.empty(n, dtype=torch.int64, device=dev), torch.empty(n, dtype=torch.int64, device=dev)
        ws = dj.workspace(L.dj_inner_join_cols_workspace_bytes(ROWS, ROWS, n), dev)
        bin_, bw = dj._col_arrays(bcols)
        pin, pw = dj._col_arrays(pcols)
        bop, pop = dj._col_arrays(bout)[0], dj._col_arrays(pout)[0]

        def cols_call():
            dj._check(L.dj_inner_join_cols(dj._ptr(bk), bin_, bw, len(bcols), ROWS, dj._ptr(pk), pin, pw, len(pcols),
                                           ROWS, dj._ptr(bko), bop, dj._ptr(pko), pop, n, dj._ptr(cnt), dj._ptr(ws),
                                           ws.numel(), st))

        cols_call()
        assert int(cnt.item()) == n
        ms, times, prof = timed(cols_call)
        widths = [c.element_size() for c in bcols + pcols]
        gather_bytes = n * sum(32 + w for w in widths) + 2 * n * 8
        gather_ms = prof["other"][0] - base_other
        line = (f"{name} dj_inner_join_cols ({'/'.join(kinds)} per side): {ms:.2f} ms median "
                f"(calls {', '.join(f'{t:.2f}' for t in times)}); "
                + ", ".join(f"{k} {v[0]:.2f} ms/{v[1]}" for k, v in prof.items())
                + f"; iota+gather {gather_ms:.2f} ms for {gather_bytes / 1e9:.1f} GB algorithmic "
                f"-> {gather_bytes / gather_ms / 1e6:.0f} GB/s")
        entry = {"ms": ms, "calls_ms": times, "profile": prof, "gather_ms": gather_ms, "gather_bytes": gather_bytes,
                 "gather_gbs": gather_bytes / gather_ms / 1e6}
        if name == "cols=1":
            ok = dj.multiset_checksum4(bko, bout[0], pko, pout[0]) == base_sum
            line += f"; checksum vs baseline: {'OK' if ok else 'MISMATCH'}"
            entry["checksum_equal_baseline"] = ok
            assert ok, "cols=1 result differs from dj_inner_join_i64"
        print(line)
        report["variants"][name] = entry
        del bcols, pcols, bout, pout, bko, pko, ws
        torch.cuda.empty_cache()
    print(json.dumps(report))


if __name__ == "__main__":
    main()
