"""Device-resident, row-sharded serving on top of the C ABI's *_dev entry points (SURVEY §8e).

One process per GPU.  The database is split by rows of the first dimension; every rank scans its rows for all ranks'
queries, re-encodes and multiplies its share of the upper dimensions and produces partial replies in NTT form.  The
partials are combined with a mod-q add (never a plain integer sum).  Two flows (setup_distributed picks one):
- NVLink (d >= 2, when every rank can map its peers' memory; pirb_dist_*): the library's own kernels store the
  selection vectors into the peers' memory and add the partial replies by peer loads;
- NCCL (otherwise): the selection vectors (for d = 1 the query ciphertexts) and the partial replies are all-gathered
  and every rank finishes its own queries with the fused add-and-inverse-NTT kernel.

torch is used only for device memory, streams and torch.distributed — uint64 limbs are carried in int64 tensors.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from .api import GaloisKeys, PIRDatabase, PIRParameters, _check, _KeyHandle

# Selection vectors of at least this many bytes per rank are exchanged split by ownership (_exchange_selection_vectors).
SPLIT_EXCHANGE_MIN_BYTES = 64 << 20


def _dp(t: torch.Tensor):
    assert t.is_cuda and t.dtype == torch.int64 and t.is_contiguous()
    return C.c_void_p(t.data_ptr())


class ShardServer:
    def __init__(self, params: PIRParameters, device=0, shard_index=0, shard_count=1):
        self.params = params
        self.device = torch.device("cuda", device)
        self.db = PIRDatabase(params, device, shard_index, shard_count)
        self.ctx = self.db.ctx
        self.shard_index, self.shard_count = shard_index, shard_count
        self.keys = None
        self._dist_mode = "nccl"
        with torch.cuda.device(self.device):
            self.stream = torch.cuda.Stream()
        self.k, self.N = self.ctx.k, self.ctx.N
        L = _lib.lib()
        self.pt_begin = int(L.pirb_shard_pt_begin(self.ctx.h))
        self.pt_count = int(L.pirb_shard_pt_count(self.ctx.h))

    # -- setup -----------------------------------------------------------------------------------
    def load_coeff(self, coeffs, first_pt=0):
        """coeffs [count][N] with GLOBAL plaintext indices starting at first_pt; the shard keeps what it owns."""
        self.db.load_coeff(coeffs, first_pt)

    def set_keys(self, gk: GaloisKeys):
        if self.keys is not None:
            self.keys.close()
        self.keys = _KeyHandle(self.ctx, gk)

    def set_profiling(self, on=True):
        _check(_lib.lib().pirb_set_profiling(self.ctx.h, 1 if on else 0))

    def stage_ms(self):
        out = (C.c_float * _lib.PIRB_N_STAGES)()
        _check(_lib.lib().pirb_get_stage_ms(self.ctx.h, out))
        return dict(zip(_lib.STAGE_NAMES, [float(x) for x in out]))

    def last_scan_ms(self):
        out = C.c_float(0)
        _check(_lib.lib().pirb_last_scan_ms(self.ctx.h, C.byref(out)))
        return float(out.value)

    def launch_count(self):
        return int(_lib.lib().pirb_last_launch_count(self.ctx.h))

    def scan_bytes(self, n_queries=1):
        return int(_lib.lib().pirb_scan_bytes(self.ctx.h, n_queries))

    # -- stream plumbing ---------------------------------------------------------------------------
    def _enter(self):
        self.stream.wait_stream(torch.cuda.current_stream(self.device))
        return C.c_void_p(self.stream.cuda_stream)

    def _exit(self):
        torch.cuda.current_stream(self.device).wait_stream(self.stream)

    def _empty(self, *shape):
        return torch.empty(shape, dtype=torch.int64, device=self.device)

    # -- hot path ----------------------------------------------------------------------------------
    def answer(self, d_queries: torch.Tensor) -> torch.Tensor:
        """[Q][n_ct][2][k][N] -> [Q][reply_cts][2][k][N] (unsharded context)."""
        Q, n_ct = d_queries.shape[0], d_queries.shape[1]
        out = self._empty(Q, self.ctx.reply_cts, 2, self.k, self.N)
        st = self._enter()
        _check(_lib.lib().pirb_answer_dev(self.ctx.h, self.keys.h if self.keys else None, _dp(d_queries), Q, n_ct,
                                          _dp(out), st))
        self._exit()
        return out

    def answer_partial(self, d_queries: torch.Tensor) -> torch.Tensor:
        """This shard's NTT-form partial replies [Q][reply_cts][2][k][N]."""
        Q, n_ct = d_queries.shape[0], d_queries.shape[1]
        out = self._empty(Q, self.ctx.reply_cts, 2, self.k, self.N)
        st = self._enter()
        _check(_lib.lib().pirb_answer_partial_dev(self.ctx.h, self.keys.h if self.keys else None, _dp(d_queries), Q,
                                                  n_ct, _dp(out), st))
        self._exit()
        return out

    def expand_ntt(self, d_queries: torch.Tensor) -> torch.Tensor:
        """Expansion + selection-vector NTT: [Q][n_ct][2][k][N] -> [Q][dim_sum][2][k][N] (NTT form)."""
        Q, n_ct = d_queries.shape[0], d_queries.shape[1]
        out = self._empty(Q, self.ctx.dim_sum, 2, self.k, self.N)
        st = self._enter()
        _check(_lib.lib().pirb_expand_ntt_dev(self.ctx.h, self.keys.h if self.keys else None, _dp(d_queries), Q, n_ct,
                                              _dp(out), st))
        self._exit()
        return out

    def multiply_partial(self, d_sv_ntt: torch.Tensor) -> torch.Tensor:
        """NTT-form selection vectors [Q][dim_sum][2][k][N] -> this shard's NTT-form partial replies."""
        Q = d_sv_ntt.shape[0]
        out = self._empty(Q, self.ctx.reply_cts, 2, self.k, self.N)
        st = self._enter()
        _check(_lib.lib().pirb_multiply_partial_dev(self.ctx.h, _dp(d_sv_ntt), Q, _dp(out), st))
        self._exit()
        return out

    def reduce_finish(self, gathered: torch.Tensor, n_queries: int) -> torch.Tensor:
        """gathered [G][Q][reply_cts][2][k][N] partials -> mod-q add + inverse NTT -> final replies."""
        G = gathered.shape[0]
        out = self._empty(n_queries, self.ctx.reply_cts, 2, self.k, self.N)
        st = self._enter()
        _check(_lib.lib().pirb_reduce_finish_dev(self.ctx.h, _dp(gathered), G, gathered[0].numel(), n_queries,
                                                 _dp(out), st))
        self._exit()
        return out

    def answer_batch_distributed(self, d_queries_local: torch.Tensor) -> torch.Tensor:
        """Batch path (SURVEY §8e): every rank expands only ITS queries, the NTT-form selection vectors are
        all-gathered, every rank multiplies ALL queries against its row shard, the partial replies are all-gathered
        and each rank finishes (mod-q add + inverse NTT) its own queries.  Returns this rank's replies."""
        import torch.distributed as dist
        world, rank = dist.get_world_size(), dist.get_rank()
        ql = d_queries_local.shape[0]
        if world > 1 and len(self.params.dimensions) == 1:
            # one-dimensional database: the selection vector is as large as the database, so it is never exchanged;
            # the (tiny) query ciphertexts are, and every rank expands only the trees that cover its own plaintexts
            q_all = self._gather_queries(d_queries_local)
            # expansion workspace per query: two ping-pong regions over this shard's trees; bound it to ~48 GB a call
            lo, hi = shard_rows(self.params.dimensions[0], self.shard_count)[self.shard_index]
            trees = max(1, (max(hi, lo + 1) - 1) // self.N - lo // self.N + 1)
            per_query = 2 * trees * self.N * 2 * self.k * self.N * 8
            chunk = max(1, (48 << 30) // per_query)
            self.last_partial_batch = (q_all.shape[0] - 1) % chunk + 1  # queries in the last library call
            part = torch.cat([self.answer_partial(q_all[i:i + chunk]) for i in range(0, q_all.shape[0], chunk)])
        else:
            sv_local = self.expand_ntt(d_queries_local)
            if world == 1:
                part = self.multiply_partial(sv_local)
                return self.reduce_finish(part[None], ql)
            sv_all = self._exchange_selection_vectors(sv_local)
            part = self.multiply_partial(sv_all)                 # [world*ql][reply_cts]...
        gathered = self._empty(world, *part.shape)
        dist.all_gather_into_tensor(gathered, part)
        own = gathered[:, rank * ql:(rank + 1) * ql]             # view: [world][ql][reply_cts]...
        out = self._empty(ql, self.ctx.reply_cts, 2, self.k, self.N)
        st = self._enter()
        _check(_lib.lib().pirb_reduce_finish_dev(self.ctx.h, C.c_void_p(own.data_ptr()), world, gathered[0].numel(),
                                                 ql, _dp(out), st))
        self._exit()
        return out

    def _gather_queries(self, d_queries_local: torch.Tensor) -> torch.Tensor:
        import torch.distributed as dist
        world = dist.get_world_size()
        q_all = self._empty(world * d_queries_local.shape[0], *d_queries_local.shape[1:])
        dist.all_gather_into_tensor(q_all, d_queries_local.contiguous())
        return q_all

    def _exchange_selection_vectors(self, sv_local: torch.Tensor) -> torch.Tensor:
        """Every rank needs, of every query: all selection ciphertexts of dimensions 1..d-1 (they multiply every row)
        but of dimension 0 only the entries of the rows it owns.  For >= 4 ranks the tail is all-gathered and the
        head is exchanged by ownership (all-to-all), which moves about half of what a full all-gather would."""
        import torch.distributed as dist
        world, rank = dist.get_world_size(), dist.get_rank()
        ql, dim_sum = sv_local.shape[0], sv_local.shape[1]
        d0 = self.params.dimensions[0]
        sv_all = self._empty(world * ql, *sv_local.shape[1:])
        # measured on 8 B200s: at 10 MB per rank (config 2) the extra all-to-all costs more latency than the halved
        # volume saves, at 85-680 MB per rank (configs 3/4) the exchange is bandwidth-bound and the split wins.
        split = sv_local.numel() * 8 >= SPLIT_EXCHANGE_MIN_BYTES
        if world < 2 or len(self.params.dimensions) == 1 or not split:
            dist.all_gather_into_tensor(sv_all, sv_local)
            return sv_all
        rows = shard_rows(d0, world)
        tail_local = sv_local[:, d0:].contiguous()
        tail_all = self._empty(world * ql, dim_sum - d0, *sv_local.shape[2:])
        dist.all_gather_into_tensor(tail_all, tail_local)
        per = sv_local[0, 0].numel()
        send = torch.cat([sv_local[:, lo:hi].reshape(-1) for lo, hi in rows])
        lo_me, hi_me = rows[rank]
        recv = self._empty(world * ql * (hi_me - lo_me) * per)
        dist.all_to_all_single(recv, send, output_split_sizes=[ql * (hi_me - lo_me) * per] * world,
                               input_split_sizes=[ql * (hi - lo) * per for lo, hi in rows])
        sv_all[:, d0:] = tail_all
        if hi_me > lo_me:
            sv_all[:, lo_me:hi_me] = recv.view(world * ql, hi_me - lo_me, *sv_local.shape[2:])
        return sv_all  # dimension-0 entries of other ranks' rows stay uninitialised: this shard never reads them

    # -- one entry point for the multi-GPU step, whatever the transport ------------------------------------------
    def setup_distributed(self, queries_per_rank: int, prefer: str = "nvlink", sub_batch: int = 0) -> str:
        """Collective.  Chooses how selection vectors and partial replies travel between the ranks and sets it up;
        returns a description for the bench line.  "nvlink": the library's own kernels store / load peer memory
        (pirb_dist_*; the process group is only used here, to swap the CUDA IPC handles).  Falls back to the NCCL flow
        (answer_batch_distributed) on every rank if any rank cannot map its peers' memory, and for one-dimensional
        databases; "nccl" always uses it."""
        import torch.distributed as dist
        world, rank = dist.get_world_size(), dist.get_rank()
        self._dist_mode = "nccl"
        if prefer == "nvlink" and len(self.params.dimensions) > 1:
            ok, err = 1, ""
            handle = (C.c_uint8 * 64)()
            try:
                _check(_lib.lib().pirb_dist_create(self.ctx.h, queries_per_rank, sub_batch, handle, None))
            except Exception as e:  # noqa: BLE001
                ok, err = 0, str(e)
            handles = [None] * world
            dist.all_gather_object(handles, bytes(handle) if ok else None)
            if all(h is not None for h in handles):
                blob = (C.c_uint8 * (64 * world)).from_buffer_copy(b"".join(handles))
                try:
                    _check(_lib.lib().pirb_dist_open_ipc(self.ctx.h, blob, world, rank))
                except Exception as e:  # noqa: BLE001
                    ok, err = 0, str(e)
            else:
                ok = 0
            flag = torch.tensor([ok], device=self.device)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if int(flag.item()):
                self._dist_mode = "nvlink"
                return ("selection vectors stored into the peers' memory by the NTT kernel, partial replies added mod q "
                        "by peer loads in the reduce kernel (NVLink, per-sub-batch flags, no collective on the data path)")
            if not ok:
                import sys
                sys.stderr.write("rank %d: peer-memory exchange unavailable (%s); using NCCL\n" % (rank, err))
        return "selection vectors and partial replies gathered with NCCL"

    def answer_dist(self, d_queries_local: torch.Tensor) -> torch.Tensor:
        """This rank's queries [ql][n_ct][2][k][N] -> this rank's replies; every rank calls it in lockstep."""
        if self._dist_mode == "nvlink":
            ql, n_ct = d_queries_local.shape[0], d_queries_local.shape[1]
            out = self._empty(ql, self.ctx.reply_cts, 2, self.k, self.N)
            st = self._enter()
            _check(_lib.lib().pirb_dist_answer_dev(self.ctx.h, self.keys.h if self.keys else None, _dp(d_queries_local),
                                                   ql, n_ct, _dp(out), st))
            self._exit()
            return out
        return self.answer_batch_distributed(d_queries_local)

    def answer_dist_host(self, q_pinned: torch.Tensor, out_pinned: torch.Tensor):
        """End-to-end variant: this rank's queries start in (pinned) host memory and its replies end there."""
        if self._dist_mode == "nvlink":
            # the C ABI's host-buffer entry point: page-locked buffers are read / written in place by the kernels
            _check(_lib.lib().pirb_dist_answer(self.ctx.h, self.keys.h if self.keys else None,
                                               C.c_void_p(q_pinned.data_ptr()), q_pinned.shape[0], q_pinned.shape[1],
                                               C.c_void_p(out_pinned.data_ptr())))
            return
        d = q_pinned.to(self.device, non_blocking=True)
        out_pinned.copy_(self.answer_dist(d), non_blocking=True)
        torch.cuda.synchronize(self.device)

    def dist_status(self):
        _check(_lib.lib().pirb_dist_status(self.ctx.h))

    def dist_stage_ms(self):
        out = (C.c_float * 10)()
        _check(_lib.lib().pirb_dist_stage_ms(self.ctx.h, out))
        return dict(zip(_lib.DIST_STAGE_NAMES, [float(x) for x in out]))

    def profile_stages(self, step, flush=None, n=5):
        """Mean per-stage device times (CUDA events recorded by the library on its launching stream) over n extra
        steps.  Profiling inserts events between kernels, so those steps run eagerly instead of as one graph."""
        self.set_profiling(True)
        acc = {}
        try:
            for _ in range(n):
                if flush is not None:
                    flush()
                step()
                torch.cuda.synchronize(self.device)
                st = self.dist_stage_ms() if self._dist_mode == "nvlink" else self.stage_ms()
                for nm, v in st.items():
                    acc.setdefault(nm, []).append(v)
        finally:
            self.set_profiling(False)
        return {nm: sum(v) / len(v) for nm, v in acc.items()}

    def scan(self, d_sv_ntt: torch.Tensor, want_rows=True):
        """[Q][dimL][2][k][N] NTT-form last-dimension selection cts -> rows [Q][n_rows][2][k][N] NTT form."""
        Q = d_sv_ntt.shape[0]
        d = len(self.params.dimensions)
        dimL = d_sv_ntt.shape[1]
        n_rows = 1 if d == 1 else -(-self.pt_count // dimL)
        out = self._empty(Q, n_rows, 2, self.k, self.N) if want_rows else None
        st = self._enter()
        _check(_lib.lib().pirb_scan_dev(self.ctx.h, _dp(d_sv_ntt), Q, _dp(out) if want_rows else None, st))
        self._exit()
        return out


class ShardGroup:
    """All row shards of one database inside ONE process: a context per shard (on `devices[i]`; several shards may share
    a device), their exchange blocks attached to each other by pointer (peer access between devices).  The same
    kernels and flags as the one-process-per-GPU flow — this is what a C++ host drives through pirb_dist_attach."""

    def __init__(self, params: PIRParameters, devices, queries_per_rank: int, sub_batch: int = 0):
        self.world = len(devices)
        self.shards = [ShardServer(params, device=d, shard_index=i, shard_count=self.world) for i, d in enumerate(devices)]
        bases = (C.c_void_p * self.world)()
        for i, sh in enumerate(self.shards):
            b = C.c_void_p()
            _check(_lib.lib().pirb_dist_create(sh.ctx.h, queries_per_rank, sub_batch, None, C.byref(b)))
            bases[i] = b.value
        for i, sh in enumerate(self.shards):
            _check(_lib.lib().pirb_dist_attach(sh.ctx.h, bases, self.world, i))
            sh._dist_mode = "nvlink"

    def fill_random(self, seed):
        for sh in self.shards:
            sh.db.fill_random(seed)

    def load_coeff(self, coeffs, first_pt=0):
        for sh in self.shards:
            sh.load_coeff(coeffs, first_pt)

    def set_keys(self, gks):
        """gks: one GaloisKeys for everybody, or one per rank (the keys of the client whose queries that rank expands)."""
        for i, sh in enumerate(self.shards):
            sh.set_keys(gks[i] if isinstance(gks, (list, tuple)) else gks)

    def answer(self, queries_per_rank):
        """queries_per_rank[i]: device tensor [ql][n_ct][2][k][N] on shard i's device -> list of reply tensors.
        Every rank's step is enqueued before anything is waited for (the ranks wait for each other on the device)."""
        # everything that may synchronise a device (allocations, first launches) happens before the first rank's step
        # is enqueued: one host thread drives all ranks, and a rank's wait kernels spin until its peers' launches exist
        outs = [sh._empty(q.shape[0], sh.ctx.reply_cts, 2, sh.k, sh.N) for sh, q in zip(self.shards, queries_per_rank)]
        for sh, q in zip(self.shards, queries_per_rank):
            _check(_lib.lib().pirb_dist_prepare(sh.ctx.h, sh.keys.h, q.shape[0]))
        for sh, q, out in zip(self.shards, queries_per_rank, outs):
            ql, n_ct = q.shape[0], q.shape[1]
            st = sh._enter()  # no join with the caller's stream until every rank's step has been enqueued
            _check(_lib.lib().pirb_dist_answer_dev(sh.ctx.h, sh.keys.h if sh.keys else None, _dp(q), ql, n_ct, _dp(out), st))
        for sh in self.shards:
            sh._exit()
        for sh in self.shards:
            torch.cuda.synchronize(sh.device)
        for sh in self.shards:
            sh.dist_status()
        return outs


def shard_rows(dim0: int, shard_count: int):
    """Row ranges [lo, hi) of dims[0] per shard — the same split the C library makes (context.cu)."""
    per = -(-dim0 // shard_count)
    return [(min(dim0, per * s), min(dim0, per * s + per)) for s in range(shard_count)]


def sampled_parity(srv: "ShardServer", orc, params, elts, keys, query: np.ndarray, reply: np.ndarray):
    """Parity of one d=2 query at sizes where the oracle cannot process the whole database: (1) the FULL expansion and
    selection-vector NTT against the oracle; (2) the scan at full size, checked on the first, a middle and the last
    (possibly short) row against the oracle's scan of those rows of the device database; (3) the upper dimension
    recomputed by the oracle (re-encode, plaintext NTT, multiply, add, inverse NTT: ct_reencoder.cpp:40-71,
    database.cpp:213-254) from ALL of the device's row results, against the reply.  srv must be unsharded.
    Returns (ok, description).  TEST INFRASTRUCTURE: the oracle is only ever the checker."""
    dims = list(params.dimensions)
    if len(dims) != 2:
        return None, "sampled parity only implemented for d=2"
    d0, dimL = dims
    dim_sum = d0 + dimL
    q = np.ascontiguousarray(query)
    d_q = to_device(q[None], srv.device)
    sv_gpu_t = srv.expand_ntt(d_q)[0]                                   # [dim_sum][2][k][N], NTT form
    sv = orc.expand(q, dim_sum, elts, np.ascontiguousarray(keys).reshape(-1))
    sv_ntt = np.stack([orc.ct_to_ntt(c) for c in sv])
    ok_exp = bool(np.array_equal(to_host(sv_gpu_t), sv_ntt))
    rows_gpu = to_host(srv.scan(sv_gpu_t[d0:][None].contiguous()))[0]   # [n_rows][2][k][N], NTT form
    n_rows = rows_gpu.shape[0]
    ok_rows = True
    picked = sorted({0, n_rows // 2, n_rows - 1})
    for r in picked:
        cnt = min(dimL, params.num_pt - r * dimL)
        db_row = srv.db.read_ntt(r * dimL, cnt)
        want = orc.scan_row(db_row, sv_ntt[d0:d0 + cnt])
        ok_rows = ok_rows and bool(np.array_equal(rows_gpu[r], want))
    two_er = reply.shape[0]
    pts = np.empty((n_rows, two_er, orc.k, orc.N), dtype=np.uint64)
    for r in range(n_rows):
        enc = orc.reencode(orc.ct_from_ntt(rows_gpu[r]))
        for x in range(two_er):
            pts[r, x] = orc.plain_to_ntt(enc[x])
    ok_up = True
    for x in range(two_er):
        acc = orc.scan_row(np.ascontiguousarray(pts[:, x]), sv_ntt[:n_rows])
        ok_up = ok_up and bool(np.array_equal(orc.ct_from_ntt(acc), reply[x]))
    desc = ("query 0 vs the oracle: full expansion + selection-vector NTT %s; scan rows %s of %d at full size %s; "
            "upper dimension recomputed by the oracle from all device rows %s" % (
                "identical" if ok_exp else "MISMATCH", picked, n_rows, "identical" if ok_rows else "MISMATCH",
                "identical" if ok_up else "MISMATCH"))
    return bool(ok_exp and ok_rows and ok_up), desc


def to_device(a: np.ndarray, device) -> torch.Tensor:
    return torch.from_numpy(np.ascontiguousarray(a).view(np.int64)).to(device)


def to_host(t: torch.Tensor) -> np.ndarray:
    return t.cpu().numpy().view(np.uint64)
