"""torchrun helper: row-sharded distributed answers must equal the oracle's answer on the whole database bit for bit.

Run as: python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tests/helpers/dist_parity.py
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import pir_b200 as pb  # noqa: E402
from oracle import client as oc  # noqa: E402
from pir_b200 import sharded  # noqa: E402


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    ok = True
    for dbsize, d in [(82, 2), (300, 2), (200, 1), (50, 3)]:
        ep = pb.GenerateEncryptionParams(4096, 20)
        p = pb.CreatePIRParameters(dbsize, 0, d, ep)
        hp = oc.PIRParameters(p.num_items, p.num_pt, list(p.dimensions), p.bytes_per_item, p.items_per_plaintext,
                              p.bits_per_coeff, ep.poly_modulus_degree, ep.plain_modulus, list(ep.coeff_modulus))
        cl = oc.HarnessClient(hp, seed=11)  # same seed on every rank -> same keys and queries
        rng = np.random.default_rng(42)
        items = [rng.integers(0, 256, p.bytes_per_item, dtype=np.uint8).tobytes() for _ in range(p.num_items)]
        coeffs = oc.encode_string_db(hp, items)
        gk = pb.GaloisKeys(cl.elts, cl.galois)
        srv = sharded.ShardServer(p, device=local, shard_index=rank, shard_count=world)
        srv.load_coeff(coeffs)
        srv.set_keys(gk)
        idxs = [(7 * r + 3) % dbsize for r in range(world)]
        queries = np.stack([cl.create_query(i) for i in idxs])          # [world][n_ct][2][k][N]
        db_ntt = oc.db_to_ntt(cl.orc, coeffs)
        want = cl.orc.process_query(db_ntt, p.dimensions, cl.elts, cl.galois, queries[rank])
        # (1) NCCL flow: rank r expands only query r
        mine = sharded.to_host(srv.answer_batch_distributed(sharded.to_device(queries[rank:rank + 1], dev)))[0]
        ok &= bool(np.array_equal(mine, want))
        # (1b) the ownership-aware exchange of the selection vectors (chosen automatically for large messages)
        split_min, sharded.SPLIT_EXCHANGE_MIN_BYTES = sharded.SPLIT_EXCHANGE_MIN_BYTES, 0
        split = sharded.to_host(srv.answer_batch_distributed(sharded.to_device(queries[rank:rank + 1], dev)))[0]
        sharded.SPLIT_EXCHANGE_MIN_BYTES = split_min
        ok &= bool(np.array_equal(split, want))
        # (2) the exchange done by the library's own kernels over peer memory (pirb_dist_*, CUDA IPC between the
        #     processes): two local queries per rank in sub-batches of one, three steps
        if d >= 2:
            nxt = (rank + 1) % world
            want_nxt = cl.orc.process_query(db_ntt, p.dimensions, cl.elts, cl.galois, queries[nxt])
            mode = srv.setup_distributed(2, prefer="nvlink", sub_batch=1)
            ok &= srv._dist_mode == "nvlink"
            two = np.stack([queries[rank], queries[nxt]])
            for _ in range(3):
                nv = sharded.to_host(srv.answer_dist(sharded.to_device(two, dev)))
                srv.dist_status()
                ok &= bool(np.array_equal(nv[0], want)) and bool(np.array_equal(nv[1], want_nxt))
            pin_q = torch.from_numpy(two.view(np.int64)).pin_memory()
            pin_r = torch.empty((2,) + nv.shape[1:], dtype=torch.int64).pin_memory()
            srv.answer_dist_host(pin_q, pin_r)                      # host-buffer entry point of the C ABI
            ok &= bool(np.array_equal(pin_r.numpy().view(np.uint64), nv))
        got = cl.process_response_strings([idxs[rank]], [mine])[0]
        ok &= got == items[idxs[rank]]
        if rank == 0:
            print("dbsize %d d=%d world=%d: %s" % (dbsize, d, world, "ok" if ok else "MISMATCH"), flush=True)
    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    dist.destroy_process_group()
    if int(flag.item()) != 1:
        sys.exit(1)
    if rank == 0:
        print("DIST_PARITY_OK")


if __name__ == "__main__":
    main()
