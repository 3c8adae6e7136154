#!/usr/bin/env python
"""Eight clients with one query each on the bench workload (BASELINE configs[3]: d=2, 2^22 x 256 B, N=4096,
fill_random), three ways:

  (a) one pirb_answer_dev per client: 8 single-query passes, each with its own scan;
  (b) one pirb_answer_multi_dev with the 8 clients' key handles: one batched pass (tensor-core scan);
  (c) one pirb_answer_dev of 8 queries under one key: bench.py's headline shape.

CUDA events around each variant, the 256 MiB L2 eviction of bench.py before each, every shape warmed first, variants
alternated step by step.  (a) and (b) must return identical replies.  Writes one JSON (--out) with the GPU name and
power limit read by nvidia-smi in the same run.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--clients", type=int, default=8)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_multi_client_cfg4.json"))
    args = ap.parse_args()

    import torch

    import bench
    import pir_b200 as pb
    from pir_b200 import _lib, sharded
    from pir_b200.api import _check, _KeyHandle
    from pir_b200.sharded import _dp

    if not torch.cuda.is_available():
        raise SystemExit("multi_client_bench.py needs a CUDA device")
    items, size, d, n, bits, desc = bench.WORKLOADS["cfg4"]
    params = pb.CreatePIRParameters(items, size, d, pb.GenerateEncryptionParams(n, bits))
    ep = params.encryption_parameters
    mods, dims = ep.coeff_modulus, list(params.dimensions)
    srv = sharded.ShardServer(params, device=0)
    srv.db.fill_random(bench.DB_SEED)
    ctx, L = srv.ctx, _lib.lib()
    Q = args.clients
    queries, elts, keys0 = bench.synth_inputs(n, mods, dims, Q, 99)
    handles = [_KeyHandle(ctx, pb.GaloisKeys(elts, keys0.reshape(-1)))]
    for c in range(1, Q):  # every client its own random Galois keys
        _, e, kc = bench.synth_inputs(n, mods, dims, 1, 1000 + c)
        handles.append(_KeyHandle(ctx, pb.GaloisKeys(e, kc.reshape(-1))))
    table = (C.c_void_p * Q)(*[h.h.value for h in handles])
    n_ct = queries.shape[1]
    d_q = sharded.to_device(queries, "cuda:0")
    shape = (Q, ctx.reply_cts, 2, ctx.k, ctx.N)
    out_a = torch.empty(shape, dtype=torch.int64, device="cuda")
    out_b = torch.empty_like(out_a)
    out_c = torch.empty_like(out_a)
    stream = torch.cuda.Stream()  # events, L2 eviction and every call on this one stream
    st = C.c_void_p(stream.cuda_stream)
    flush = torch.zeros(256 << 20, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()

    def run_a():
        for i in range(Q):
            _check(L.pirb_answer_dev(ctx.h, handles[i].h, _dp(d_q[i:i + 1]), 1, n_ct, _dp(out_a[i:i + 1]), st))

    def run_b():
        _check(L.pirb_answer_multi_dev(ctx.h, table, _dp(d_q), Q, n_ct, _dp(out_b), st))

    def run_c():
        _check(L.pirb_answer_dev(ctx.h, handles[0].h, _dp(d_q), Q, n_ct, _dp(out_c), st))

    variants = {"a_per_client": run_a, "b_multi": run_b, "c_one_key": run_c}
    torch.cuda.set_stream(stream)
    for _ in range(max(3, args.warmup)):
        for fn in variants.values():
            flush.view(torch.int64).sum()
            fn()
    torch.cuda.synchronize()
    ev = {k: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
          for k in variants}
    for s in range(args.steps):
        for k, fn in variants.items():
            flush.view(torch.int64).sum()
            ev[k][s][0].record()
            fn()
            ev[k][s][1].record()
    torch.cuda.synchronize()
    assert torch.equal(out_a, out_b), "(a) and (b) differ"
    ms = {k: [a.elapsed_time(b) for a, b in v] for k, v in ev.items()}
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    res = {
        "workload": desc,
        "clients": Q,
        "gpu": smi[0] if smi else "unknown",
        "steps": args.steps,
        "method": "CUDA events around each variant on the launching stream; 256 MiB read between variants evicts L2; "
                  "variants alternated step by step after %d warm-ups" % max(3, args.warmup),
        "replies_a_equal_b": True,
    }
    for k, v in ms.items():
        a = np.array(v)
        res[k] = {"mean_ms": float(a.mean()), "median_ms": float(np.median(a)), "min_ms": float(a.min()),
                  "max_ms": float(a.max()), "std_ms": float(a.std()), "queries_per_s": float(Q / (np.median(a) / 1e3))}
    res["b_over_c_median"] = res["b_multi"]["median_ms"] / res["c_one_key"]["median_ms"]
    res["a_over_b_median"] = res["a_per_client"]["median_ms"] / res["b_multi"]["median_ms"]
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
