"""Kernel time of the nearest-neighbour search (c2v_nearest) at the java14m table shapes.

    python tools/similarity_bench.py [--reps 20] [--out profiles/r03_similarity_bench.json]

Banks: the target table (261,246 x 384, 401 MB) and the token table (1,301,137 x 128, 666 MB), random fp32; both are
larger than the 126 MB L2, so repeated passes read HBM.  Queries: n = 1, 8, 64, 1024 at k = 10.  Each case is warmed
up, then timed with CUDA events around `reps` back-to-back calls (query chunking, candidate scratch and the merge
included; scratch allocated once outside the window).  Reported per case: ms per call, the bytes and FMAs the
algorithm needs (bytes = rows * dim * 4 per query chunk, FMAs = rows * dim * n for the dots plus rows * dim per query
chunk for the row norms), achieved GB/s, and the share of whichever bound is larger: HBM at 7.7 TB/s or fp32 FFMA at
148 SMs x 128 lanes x the card's maximum SM clock.  The device name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

HBM_BYTES_PER_S = 7.7e12
BANKS = {"target": (261246, 384), "token": (1301137, 128)}


def device_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"device": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as exc:          # the numbers stay valid; only the label is missing
        return {"device": "unknown (%s)" % exc, "power_limit": "unknown", "max_sm_clock": "unknown"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from code2vec_b200.engine import EngineDims, PathAttentionEngine
    if not torch.cuda.is_available():
        raise SystemExit("similarity_bench needs a CUDA device")
    info = device_info()
    clock_mhz = float(info["max_sm_clock"].split()[0]) if info["max_sm_clock"][:1].isdigit() else 1965.0
    fma_per_s = torch.cuda.get_device_properties(0).multi_processor_count * 128 * clock_mhz * 1e6
    eng = PathAttentionEngine(EngineDims(16, 16, 16, 4, 4, 4, 4, 4), device=0, training=False)
    g = torch.Generator(device="cuda")
    g.manual_seed(0)
    results = []
    for bank_name, (rows, dim) in BANKS.items():
        bank = torch.randn((rows, dim), generator=g, device="cuda", dtype=torch.float32)
        for n in (1, 8, 64, 1024):
            queries = torch.randn((n, dim), generator=g, device="cuda", dtype=torch.float32)
            nbytes = int(eng.lib.c2v_nearest_scratch_bytes(rows, n, args.k))
            scratch = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
            idx = torch.empty((n, args.k), dtype=torch.int32, device="cuda")
            val = torch.empty((n, args.k), dtype=torch.float32, device="cuda")

            def call():
                eng._check(eng.lib.c2v_nearest(eng.h, bank.data_ptr(), rows, dim, queries.data_ptr(), n, args.k, None, 0,
                                               idx.data_ptr(), val.data_ptr(), scratch.data_ptr(), nbytes,
                                               eng._stream()))
            for _ in range(3):
                call()
            torch.cuda.synchronize()
            start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            start.record()
            for _ in range(args.reps):
                call()
            end.record()
            torch.cuda.synchronize()
            ms = start.elapsed_time(end) / args.reps
            chunks = (n + PathAttentionEngine.nearest_query_capacity(dim) - 1) // PathAttentionEngine.nearest_query_capacity(dim)
            need_bytes = rows * dim * 4 * chunks
            need_fma = rows * dim * (n + chunks)
            t_bytes, t_fma = need_bytes / HBM_BYTES_PER_S, need_fma / fma_per_s
            bound = "hbm" if t_bytes >= t_fma else "fp32_fma"
            r = {"bank": bank_name, "rows": rows, "dim": dim, "n": n, "k": args.k, "query_chunks": chunks,
                 "ms": round(ms, 4), "bytes": need_bytes, "fma": need_fma,
                 "achieved_GBps": round(need_bytes / (ms * 1e-3) / 1e9, 1),
                 "achieved_TFMAps": round(need_fma / (ms * 1e-3) / 1e12, 2),
                 "bound": bound, "share_of_bound": round(max(t_bytes, t_fma) / (ms * 1e-3), 3)}
            results.append(r)
            print(json.dumps(r), flush=True)
        del bank
    report = dict(info, reps=args.reps, hbm_peak_TBps=HBM_BYTES_PER_S / 1e12,
                  fp32_fma_peak_TFMAps=round(fma_per_s / 1e12, 2), results=results)
    print(json.dumps({k: v for k, v in report.items() if k != "results"}))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(report, f, indent=1)
    eng.close()


if __name__ == "__main__":
    main()
