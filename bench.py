#!/usr/bin/env python
"""bench.py — PIR server answer path on B200 (BASELINE.json metric: queries/sec + p50 latency + DB-scan GB/s).

Default workload (config.workload): BASELINE.json configs[3] — d=2, 2^22 elements x 256 B, BFV N=4096 (110 377
plaintexts, dims [333,332], 6.74 GiB NTT-form database, 1023 key switches and 8 reply ciphertexts per query), a batch
of 8 concurrent queries per GPU sharing one database scan (64 on 8 GPUs = configs[3] verbatim).  A step = one pass of
the hot path (oblivious expansion + database multiply, server.cpp:173-195) over one batch of queries:
  N=1  : 8 queries against the whole database on one GPU;
  N>1  : 8 queries per GPU per step (weak scaling).  The database is row-sharded across the N GPUs; each rank expands
         its own queries, the NTT-form selection vectors reach the peers over NVLink, every rank multiplies all 8N
         queries against its rows, partial replies are combined with a mod-q add over peer memory.
Synthetic data: uniform limbs in [0,q_j) for the NTT-form database (generated on the device from a counter-based
hash of the GLOBAL limb index, so shards are slices of the unsharded database), query ciphertexts and Galois keys
(every kernel on the path is data-independent).  `value` is device-resident throughput (inputs already in HBM); `e2e`
goes through the reference-facing call (PIRServer.ProcessRequest -> C ABI pirb_answer) with pinned HOST buffers,
H2D/D2H inside, matching what pir/cpp/benchmark.cpp:71-79 times minus (de)serialization.
`roofline` is the single-query database scan (k_scan, the HBM-bound kernel) on this GPU's share of that database,
timed live with CUDA events on its launching stream.  `latency_cfg2` (N=1 only) is the single-query latency on
BASELINE configs[1] (the configuration round 1 was quoted on).

--impl reference times the CPU restatement of the reference path (oracle/, SEAL-3.5.6-equivalent algorithms; SEAL itself
cannot be built here) on all host threads for the same workload.  That arm never imports pir_b200.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (num_items, bytes_per_item, dims, N, plain_bits, description)
    "cfg4": (1 << 22, 256, 2, 4096, 20, "d=2, 2^22 x 256 B, N=4096 (BASELINE configs[3])"),
    "cfg2": (1 << 16, 288, 2, 4096, 24, "d=2, 2^16 x 288 B, N=4096, t 24-bit (BASELINE configs[1])"),
    "cfg1": (4096, 64, 1, 4096, 20, "d=1, 4096 x 64 B, N=4096 (BASELINE configs[0])"),
    "cfg3": (1 << 20, 1024, 2, 8192, 20, "d=2, 2^20 x 1 KiB, N=8192 (BASELINE configs[2] database)"),
    "cfg5a": (1 << 24, 256, 1, 4096, 20, "d=1, 2^24 x 256 B, N=4096 (BASELINE configs[4], d=1 arm)"),
    "cfg5b": (1 << 24, 256, 2, 4096, 20, "d=2, 2^24 x 256 B, N=4096 (BASELINE configs[4], d=2 arm)"),
}
DEFAULT_QUERIES_PER_GPU = {"cfg4": 8}
DB_SEED = 2024
DUMP_LIMIT_BYTES = 64 * 10 ** 6  # --dump-outputs, over all ranks
DUMP_SEED = 7


def workload_string(name, ql, world):
    desc = WORKLOADS[name][5]
    if ql == 1:
        return desc + ", one query per GPU per step"
    return desc + ", %d concurrent queries per GPU sharing one DB scan (%d per step)" % (ql, ql * world)


def random_limbs(rng, moduli, shape_prefix, N):
    """uniform [*shape_prefix][len(moduli)][N] with limb j < moduli[j]"""
    out = np.empty(tuple(shape_prefix) + (len(moduli), N), dtype=np.uint64)
    for j, q in enumerate(moduli):
        out[..., j, :] = rng.integers(0, int(q), size=tuple(shape_prefix) + (N,), dtype=np.uint64)
    return out


def synth_inputs(N, mods, dims, n_queries, seed):
    k = len(mods) - 1
    rng = np.random.default_rng(seed)
    n_ct = sum(dims) // N + 1
    queries = random_limbs(rng, mods[:k], (n_queries, n_ct, 2), N)                 # [Q][n_ct][2][k][N]
    elts = [(N >> i) + 1 for i in range(N.bit_length() - 1)]
    keys = random_limbs(rng, mods, (len(elts), k, 2), N)                           # [n][k][2][k+1][N]
    return queries, elts, keys


def dump_replies(out_dir, name, replies, limit_bytes):
    """out_dir/<name>.npy, a file of at most limit_bytes: the uint64 reply limbs as float64, exact because every limb is
    below its < 2^53 modulus.  When the whole array does not fit, a seeded sample of flat positions in increasing order,
    the same for every run of that shape."""
    if replies.size and int(replies.max()) >= 1 << 53:
        raise SystemExit("--dump-outputs: reply limbs of 53 bits or more have no exact float64 form")
    vals = replies.astype(np.float64)
    n = (limit_bytes - 4096) // vals.itemsize  # 4 KiB kept for the .npy header (128 bytes for these shapes)
    if vals.size > n:
        pick = np.random.default_rng(DUMP_SEED).choice(vals.size, n, replace=False)
        vals = vals.reshape(-1)[np.sort(pick)]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), vals)


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region, from the enqueuing thread itself: all timed steps
    are enqueued first (the host runs ahead of the GPU), then NVML is polled until the last step's end event has
    completed.  NVML queries take a driver lock that can stall kernel launches for milliseconds, so they must not run
    concurrently with the enqueue loop (a sampling thread did exactly that and added 4-9 ms to single steps)."""

    def __init__(self, gpu_index):
        # NVML enumerates physical devices; honour a CUDA_VISIBLE_DEVICES remap of numeric indices
        vis = [v for v in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if v.strip().isdigit()]
        self.idx = int(vis[gpu_index]) if gpu_index < len(vis) else gpu_index
        self.sm, self.mx, self.reasons = [], None, set()
        self.nv = None
        try:
            import pynvml as nv
            nv.nvmlInit()
            self.nv = nv
            self.h = nv.nvmlDeviceGetHandleByIndex(self.idx)
            self.mx = float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM))
            self.names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                          "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                          "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                          "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
            self.get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                nv.nvmlDeviceGetCurrentClocksThrottleReasons
            self._sample()      # resolves every NVML entry point now, outside the timed region
            self.sm = []
        except Exception as e:  # noqa: BLE001
            self.nv = None
            self.reasons.add("nvml unavailable: %s" % type(e).__name__)

    def _sample(self):
        self.sm.append(float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
        r = self.get_reasons(self.h)
        for nm, bit in self.names.items():
            if r & bit:
                self.reasons.add(nm)

    def sample_until(self, done_event):
        """Poll while the GPU is still working through the enqueued timed steps (at least one sample)."""
        if self.nv is None:
            return
        try:
            while True:
                self._sample()
                if done_event.query():
                    break
                time.sleep(0.0005)
        except Exception as e:  # noqa: BLE001
            self.reasons.add("nvml unavailable: %s" % type(e).__name__)

    def result(self):
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.mx,
                "reasons": sorted(self.reasons), "samples": len(self.sm)}


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# =====================================================================================================
def run_reference(args):
    """Reference arm: the CPU restatement of the reference's path on all host threads (rank 0 only).  Nothing of
    pir_b200 is imported here: shapes come from the oracle's own restatement of parameters.cpp."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from concurrent.futures import ThreadPoolExecutor
    from oracle import binding as ob
    from oracle import client as oc
    items, size, d, n, bits, _ = WORKLOADS[args.workload]
    hp = oc.create_pir_parameters(items, size, d, N=n, plain_bits=bits)
    N, mods, dims, num_pt = hp.poly_modulus_degree, hp.coeff_modulus, list(hp.dimensions), hp.num_pt
    k = len(mods) - 1
    cores = os.cpu_count() or 1
    orc = ob.Oracle(N, mods, hp.plain_modulus)
    rng = np.random.default_rng(1234)
    ql = args.queries_per_gpu
    # bounded sample of the workload when the database does not fit a sane host allocation: keep the first rows of the
    # hypercube (whole rows), time expansion and multiply separately and scale the multiply by rows
    host_cap = int(os.environ.get("PIRB_REF_HOST_CAP_MB", 8192)) << 20
    rows_total = -(-num_pt // dims[-1]) if d > 1 else 1
    sampled = d > 1 and num_pt * k * N * 8 > host_cap
    if sampled:
        rows_s = max(1, host_cap // (dims[-1] * k * N * 8))
        db = random_limbs(rng, mods[:k], (rows_s * dims[-1],), N)
        sample = ("expansion in full + multiply against the first %d of %d rows of the database, multiply time scaled "
                  "by rows" % (rows_s, rows_total))
    else:
        db = random_limbs(rng, mods[:k], (num_pt,), N)
        sample = "full workload"
    queries, elts, keys = synth_inputs(N, mods, dims, cores, 99)
    keys = keys.reshape(-1)

    def one(i):
        """-> estimated seconds of ProcessRequest-equivalent work (expansion + multiply) for one full query"""
        q = queries[i % len(queries)]
        t0 = time.perf_counter()
        if not sampled:
            orc.process_query(db, dims, elts, keys, q)
            return time.perf_counter() - t0
        sv = orc.expand(q, sum(dims), elts, keys)
        t1 = time.perf_counter()
        sv_s = np.concatenate([sv[:rows_s], sv[dims[0]:]])
        orc.db_multiply(db, [rows_s] + dims[1:], sv_s)
        t2 = time.perf_counter()
        return (t1 - t0) + (t2 - t1) * rows_total / rows_s

    pool = ThreadPoolExecutor(cores)
    t_one = one(0)
    # a step = `cores` concurrent queries, one per thread
    for _ in range(args.warmup):
        list(pool.map(one, range(cores)))
    est, wall = [], []
    for _ in range(args.steps):
        s0 = time.perf_counter()
        est.extend(pool.map(one, range(cores)))
        wall.append(time.perf_counter() - s0)
    if sampled:
        # every thread ran one (partly scaled) query concurrently: throughput = threads / mean estimated query time
        step_s = statistics.mean(est)
    else:
        step_s = statistics.mean(wall)
    qps = cores / step_s
    line = {
        "impl": "reference", "metric": "pir_queries_per_sec", "value": qps, "unit": "queries/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * step_s,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": workload_string(args.workload, ql, max(1, args.gpus)), "queries_per_step": cores,
                   "num_pt": num_pt, "dims": dims},
        "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": cores, "kind": "port",
                         "sample": sample + "; %d concurrent queries per step, one per host thread (the GPU arm's %d "
                                            "queries per GPU do not fill the host's threads)" % (cores, ql),
                         "single_query_latency_ms": 1e3 * t_one},
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "CPU restatement of the reference path (SEAL 3.5.6 algorithms; SEAL itself is not buildable offline)",
    }
    print(json.dumps(line))


# =====================================================================================================
def run_ours(args):
    import torch
    import torch.distributed as dist

    import pir_b200 as pb
    from pir_b200 import sharded

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus must equal WORLD_SIZE")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    items, size, d, n, bits, _ = WORKLOADS[args.workload]
    params = pb.CreatePIRParameters(items, size, d, pb.GenerateEncryptionParams(n, bits))
    ep = params.encryption_parameters
    N, mods = ep.poly_modulus_degree, ep.coeff_modulus
    dims = list(params.dimensions)
    k = len(mods) - 1
    ctL = 2 * k * N
    srv = sharded.ShardServer(params, device=local_rank, shard_index=rank, shard_count=world)
    srv.db.fill_random(DB_SEED)
    ql = args.queries_per_gpu
    queries, elts, keys = synth_inputs(N, mods, dims, world * ql, 99)
    gk = pb.GaloisKeys(elts, keys.reshape(-1))
    srv.set_keys(gk)
    n_ct = queries.shape[1]
    q_local = queries[rank * ql:(rank + 1) * ql]
    d_q = sharded.to_device(q_local, dev)
    flush = torch.zeros(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def flush_l2():
        # read (not write) a buffer larger than L2: everything of ours is evicted and only CLEAN lines are left behind,
        # so the timed step does not also pay for writing back 126 MB of dirty flush data
        return flush.view(torch.int64).sum()

    mode = "single GPU"
    if world > 1:
        mode = srv.setup_distributed(ql, prefer=args.exchange)

    def step_dev():
        if world == 1:
            return srv.answer(d_q)
        return srv.answer_dist(d_q)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---------------- device-resident throughput ----------------
    out = None
    for _ in range(max(3, args.warmup)):
        flush_l2()
        out = step_dev()  # held like in the timed loop, so the caching allocator already owns both reply buffers
    sampler = ClockSampler(local_rank) if rank == 0 else None
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for i in range(args.steps):
        flush_l2()  # L2 flush between timed iterations, outside the per-step events
        ev[i][0].record()
        out = step_dev()
        ev[i][1].record()
    if sampler is not None:
        sampler.sample_until(ev[-1][1])  # clocks under load: the queue of timed steps is still executing
    barrier()
    clocks = sampler.result() if sampler is not None else None
    launches = srv.launch_count() * args.steps
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms.item())
    qps = world * ql * args.steps / (total_ms / 1e3)
    reply_dev = out.clone()

    # per-stage device times (CUDA events recorded by the library on its launching stream), measured live on
    # extra steps: profiling inserts events between kernels, so those steps run eagerly instead of as one graph
    stage_mean = srv.profile_stages(step_dev, flush_l2, args.steps)

    # ---------------- roofline: the single-query database scan on this GPU's rows, timed live ----------------
    dimL = dims[-1] if d > 1 else None
    scan_ms, scan_bytes = None, None
    if d > 1:
        rng = np.random.default_rng(5)
        sv1 = sharded.to_device(random_limbs(rng, mods[:k], (1, dimL, 2), N), dev)
        srv.set_profiling(True)
        ts = []
        for i in range(3 + args.steps):
            flush_l2()
            srv.scan(sv1, want_rows=False)
            torch.cuda.synchronize()
            if i >= 3:
                ts.append(srv.last_scan_ms())
        srv.set_profiling(False)
        scan_ms = statistics.mean(ts)
        scan_bytes = srv.scan_bytes(1)
        del sv1

    # ---------------- end to end through the reference-facing call, host buffers ----------------
    q_pin = torch.empty(q_local.shape, dtype=torch.int64).pin_memory()
    q_pin.copy_(torch.from_numpy(q_local.view(np.int64)))
    out_pin = torch.empty((ql, srv.ctx.reply_cts, 2, k, N), dtype=torch.int64).pin_memory()
    q_np = q_pin.numpy().view(np.uint64)
    out_np = out_pin.numpy().view(np.uint64)
    if world == 1:
        server = pb.PIRServer(srv.db, params)
        req = pb.Request([q_np[i] for i in range(ql)], gk)

        def step_e2e():
            server.ProcessRequest(req, out=out_np)  # H2D + kernels + D2H + sync inside pirb_answer
    else:
        def step_e2e():
            srv.answer_dist_host(q_pin, out_pin)    # pinned host -> device, distributed step, device -> pinned host, sync

    for _ in range(3):
        step_e2e()
    barrier()
    lat = []
    t0 = time.perf_counter()
    for _ in range(args.steps):
        s0 = time.perf_counter()
        step_e2e()
        lat.append(time.perf_counter() - s0)
    barrier()
    e2e_total = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_total, op=dist.ReduceOp.MAX)
    e2e_qps = world * ql * args.steps / float(e2e_total.item())
    e2e_same = bool(np.array_equal(out_np, sharded.to_host(reply_dev)))
    if args.dump_outputs:
        # the replies of the last timed step, [queries of this rank][reply_cts][2][k][N], as the caller receives them
        dump_replies(args.dump_outputs, "replies" if world == 1 else "replies_rank%d" % rank,
                     sharded.to_host(reply_dev), DUMP_LIMIT_BYTES // world)

    # ---------------- parity: the timed path against the CPU oracle (and, sharded, against the unsharded GPU path) ---
    parity, parity_detail, cpu = None, None, None
    if not args.no_parity:
        db_bytes = params.num_pt * k * N * 8
        ref_srv = srv
        ok_local = 1
        if world > 1:
            # every rank: its own replies from the row-sharded flow == the unsharded answer on this GPU
            ref_srv = sharded.ShardServer(params, device=local_rank, shard_index=0, shard_count=1)
            ref_srv.db.fill_random(DB_SEED)
            ref_srv.set_keys(gk)
            ok_local = int(torch.equal(ref_srv.answer(d_q), reply_dev))
            flag = torch.tensor([ok_local], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            ok_all = int(flag.item())
        else:
            ok_all = 1
        if rank == 0:
            from oracle import binding as ob
            orc = ob.Oracle(N, mods, ep.plain_modulus)
            if db_bytes <= (10 << 30):
                db_host = ref_srv.db.read_ntt(0, params.num_pt)
                t0 = time.perf_counter()
                want = orc.process_query(db_host, dims, elts, keys.reshape(-1), q_local[0])
                ts = [time.perf_counter() - t0]
                ok_oracle = bool(np.array_equal(sharded.to_host(reply_dev[0]), want))
                parity_detail = "reply of query 0 vs oracle.process_query on the full database: %s" % (
                    "identical" if ok_oracle else "MISMATCH")
                if world == 1 and not args.no_cpu_baseline:
                    while sum(ts) < 12.0 and len(ts) < 5:
                        t0 = time.perf_counter()
                        orc.process_query(db_host, dims, elts, keys.reshape(-1), q_local[len(ts) % ql])
                        ts.append(time.perf_counter() - t0)
                    med = statistics.median(ts)
                    cpu = {"value": 1.0 / med, "unit": "queries/s", "cores": 1, "kind": "port",
                           "sample": "%d full queries of this workload (expansion + multiply against the whole database) "
                                     "on one host thread, median" % len(ts),
                           "p50_latency_ms": 1e3 * med, "host_cpus": os.cpu_count()}
                del db_host
            else:
                # database too large for a host copy: full expansion + multiply against the first and the last rows
                ok_oracle, parity_detail = sharded.sampled_parity(ref_srv, orc, params, elts, keys, q_local[0],
                                                                  sharded.to_host(reply_dev[0]))
            parity = bool(ok_oracle and ok_all)
            if world > 1:
                parity_detail += "; every rank's replies vs the unsharded GPU answer of the same queries: %s" % (
                    "identical" if ok_all else "MISMATCH")
        if ref_srv is not srv:
            del ref_srv

    # ---------------- N=1: the C++ drop-in itself (pir::PIRServer::ProcessRequest of the shim), limbs and wire bytes ----
    shim = None
    if world == 1 and not args.no_shim:
        shim = run_shim_bench(items, size, d, n, bits, ql, args.steps)

    # ---------------- N=1: single-query latency on BASELINE configs[1] ----------------
    latency_cfg2 = None
    if world == 1 and args.workload != "cfg2" and not args.no_cfg2:
        latency_cfg2 = cfg2_latency(pb, sharded, torch, dev, local_rank, flush_l2, args.steps)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = measured_peak()
    roofline = None
    if scan_ms:
        achieved = scan_bytes / (scan_ms * 1e-3) / 1e9
        traffic, traffic_src = args.scan_traffic, "--scan-traffic"
        if traffic is None and world == 1:
            try:  # dram__bytes_read.sum + dram__bytes_write.sum of one scan launch, from the committed ncu --set full capture
                with open(os.path.join(ROOT, "profiles", "r2_scan_traffic.json")) as f:
                    t = json.load(f)
                if t.get("workload") == args.workload:
                    traffic, traffic_src = t["traffic_bytes"], "ncu --set full capture committed as profiles/" + t.get("source", "r2_scan_traffic.json")
            except Exception:  # noqa: BLE001
                traffic = None
        roofline = {"kernel": "k_scan", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src if traffic else None,
                    "peak_source": peak_src, "bytes_per_launch": scan_bytes, "ms_per_launch": scan_ms,
                    "what": "single-query scan of this GPU's rows of the database (%d plaintexts), %d launches after 3 "
                            "warm-ups, CUDA events on the launching stream, L2 flushed between launches" % (
                                srv.pt_count, args.steps)}

    # ---------------- expansion (FP64-pipe-bound): algorithmic FP64 operations of the key switches / stage time -----
    # per key switch: k(k+1) forward + 2(k+1) inverse transforms of N/2*log2(N) butterflies at 8 FP64 ops, 2k(k+1)N
    # digit-key products at 8, canonicalisation of the k(k+1) digit transforms at 4 per coefficient, the final
    # psi^-i/N scaling of the 2(k+1) inverse transforms at 7, the mod-down of 2k polynomials at 20 (DESIGN.md §4.2)
    logn = N.bit_length() - 1
    ks_per_query = sum(int(pb.next_power_two(min(N, max(0, sum(dims) - t * N)))) - 1 for t in range(n_ct))
    ops_per_ks = ((k * (k + 1) + 2 * (k + 1)) * (N // 2) * logn * 8 + 2 * k * (k + 1) * N * 8 + k * (k + 1) * N * 4
                  + 2 * (k + 1) * N * 7 + 2 * k * N * 20)
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    fp64_peak = 57.7 * torch.cuda.get_device_properties(dev).multi_processor_count * sm_mhz * 1e6 / 1e12
    expansion = None
    if stage_mean and stage_mean.get("expand"):
        exp_ms = stage_mean["expand"]
        exp_ach = ql * ks_per_query * ops_per_ks / (exp_ms * 1e-3) / 1e12
        expansion = {"kernel": "k_ks_level_cluster", "bound": "fp64 pipe", "key_switches_per_step": ql * ks_per_query,
                     "fp64_ops_per_key_switch": ops_per_ks, "achieved": exp_ach, "peak": fp64_peak, "unit": "T FP64 op/s",
                     "frac": exp_ach / fp64_peak, "ms": exp_ms,
                     "peak_source": "57.7 DFMA/clk/SM measured with tools/pipe_bench.cu x SM count x SM clock under load"}

    line = {
        "metric": "pir_queries_per_sec", "value": qps, "unit": "queries/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": total_ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": workload_string(args.workload, ql, world), "queries_per_step": world * ql,
                   "num_pt": params.num_pt, "dims": dims, "key_switches_per_query": ks_per_query,
                   "reply_cts": srv.ctx.reply_cts,
                   "parallelism": "rows sharded x%d, expansion split by query; %s" % (world, mode),
                   "l2": "256 MiB buffer read between timed iterations (evicts L2, leaves clean lines; outside the per-step CUDA events)",
                   "galois_keys": "resident in HBM, uploaded once per client"},
        "p50_latency_ms": statistics.median(step_ms),
        "step_ms": [round(x, 4) for x in step_ms],
        "e2e": {"value": e2e_qps, "unit": "queries/s", "h2d_bytes_per_step": int(world * ql * n_ct * ctL * 8),
                "d2h_bytes_per_step": int(world * ql * srv.ctx.reply_cts * ctL * 8),
                "p50_latency_ms": 1e3 * statistics.median(lat), "replies_equal_device_path": e2e_same,
                "transfer": ("PIRServer.ProcessRequest -> pirb_answer with pinned host buffers: the first kernel reads "
                             "the queries and the last one writes the replies over PCIe in place, inside the timed "
                             "region") if world == 1 else
                            "pinned host buffers, H2D of this rank's queries and D2H of its replies inside every step"},
        "gpu_launches": int(launches),
        "roofline": roofline,
        "expansion": expansion,
        "stages_ms": stage_mean,
        "cpu_baseline": cpu,
        "parity_vs_oracle": parity,
        "parity": parity_detail,
        "latency_cfg2": latency_cfg2,
        "e2e_cpp": (shim or {}).get("e2e_cpp"),
        "e2e_wire": (shim or {}).get("e2e_wire"),
        "clocks": clocks,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_shim_bench(items, size, d, n, bits, nq, steps, n_gpus=1):
    """build/shim_bench: the same workload through the C++ shim's PIRServer::ProcessRequest, in its own process."""
    import subprocess
    exe = os.path.join(ROOT, "build", "shim_bench")
    if not os.path.exists(exe):
        return {"e2e_cpp": {"unavailable": "build/shim_bench not built"}, "e2e_wire": None}
    try:
        out = subprocess.run([exe, str(items), str(size), str(d), str(n), str(bits), str(nq), str(steps), str(n_gpus)],
                             capture_output=True, text=True, timeout=600)
        return json.loads(out.stdout.strip().splitlines()[-1])
    except Exception as e:  # noqa: BLE001
        return {"e2e_cpp": {"unavailable": "%s: %s" % (type(e).__name__, e)}, "e2e_wire": None}


def cfg2_latency(pb, sharded, torch, dev, local_rank, flush_l2, steps):
    """Single-query latency on BASELINE configs[1] (d=2, 2^16 x 288 B): device-resident and through ProcessRequest."""
    items, size, d, n, bits, desc = WORKLOADS["cfg2"]
    params = pb.CreatePIRParameters(items, size, d, pb.GenerateEncryptionParams(n, bits))
    ep = params.encryption_parameters
    N, mods = ep.poly_modulus_degree, ep.coeff_modulus
    k = len(mods) - 1
    srv = sharded.ShardServer(params, device=local_rank)
    srv.db.fill_random(DB_SEED)
    queries, elts, keys = synth_inputs(N, mods, list(params.dimensions), 1, 99)
    gk = pb.GaloisKeys(elts, keys.reshape(-1))
    srv.set_keys(gk)
    d_q = sharded.to_device(queries, dev)
    for _ in range(5):
        flush_l2()
        srv.answer(d_q)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    torch.cuda.synchronize()
    for i in range(steps):
        flush_l2()
        ev[i][0].record()
        srv.answer(d_q)
        ev[i][1].record()
    torch.cuda.synchronize()
    ms = [a.elapsed_time(b) for a, b in ev]
    stages = srv.profile_stages(lambda: srv.answer(d_q), flush_l2, steps)
    q_pin = torch.from_numpy(queries.view(np.int64)).pin_memory()
    out_pin = torch.empty((1, srv.ctx.reply_cts, 2, k, N), dtype=torch.int64).pin_memory()
    server = pb.PIRServer(srv.db, params)
    req = pb.Request([q_pin.numpy().view(np.uint64)[0]], gk)
    out_np = out_pin.numpy().view(np.uint64)
    for _ in range(5):
        server.ProcessRequest(req, out=out_np)
    lat = []
    for _ in range(steps):
        s0 = time.perf_counter()
        server.ProcessRequest(req, out=out_np)
        lat.append(time.perf_counter() - s0)
    return {"workload": desc + ", one query", "p50_ms": statistics.median(ms), "queries_per_s": 1e3 * steps / sum(ms),
            "e2e_p50_ms": 1e3 * statistics.median(lat), "e2e_queries_per_s": steps / sum(lat), "stages_ms": stages,
            "steps": steps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of every timed loop: the headline device loop, the end-to-end loop, the per-stage "
                         "profile, the k_scan roofline launches, the C++ shim bench, the cfg2 latency and the reference "
                         "arm; only the single-thread CPU baseline keeps its own bound (up to 5 oracle queries or 12 s)")
    ap.add_argument("--warmup", type=int, default=3,
                    help="untimed steps before the headline loop (the GPU arm runs at least 3: the second call of a "
                         "shape captures its CUDA graph, the third replays it)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg4", choices=sorted(WORKLOADS))
    ap.add_argument("--queries-per-gpu", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-cfg2", action="store_true")
    ap.add_argument("--no-shim", action="store_true")
    ap.add_argument("--exchange", default="nvlink", choices=["nvlink", "nccl"],
                    help="N>1: selection vectors and partial replies travel by in-kernel NVLink peer stores/loads "
                         "(default) or by NCCL all-gather")
    ap.add_argument("--scan-traffic", type=float, default=None,
                    help="dram bytes per scan launch; default: the committed ncu capture in profiles/ for this workload")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the replies of the last one to DIR/replies.npy (with --gpus > 1, "
                         "DIR/replies_rank<r>.npy per rank) as exact float64, at most 64 MB in all; the inputs are seeded, "
                         "so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the replies of the GPU path; --impl reference has none")
    if args.queries_per_gpu is None:
        args.queries_per_gpu = DEFAULT_QUERIES_PER_GPU.get(args.workload, 1)
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        if args.impl == "reference":
            run_reference(args)
            return
        # convenience: `python bench.py --gpus N` re-launches itself as one rank per GPU (the driver's own launch line)
        import socket
        with socket.socket() as sk:
            sk.bind(("127.0.0.1", 0))
            port = sk.getsockname()[1]
        os.execvp(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                                   "--nproc-per-node", str(args.gpus), "--master-addr", "127.0.0.1",
                                   "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:])
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
