"""Queries of several clients, each with its own Galois keys, answered in one batched pass (pirb_answer_multi*,
PIRServer.ProcessRequests in Python and C++).

Only the expansion reads the keys: every key-switch kernel takes query qi's key from a per-level table of key pointers
(LevelArgs.key_tab).  The tests check, limb for limb, that a batch of mixed clients answers every request exactly as
that request alone does (ProcessRequest) and as the CPU oracle does with that client's keys; that real clients decrypt
their items; that every key-switch implementation picks the right key for each query; that the captured graphs serve
any mix of clients; that a bad handle is rejected before anything runs; and that the key caches never free keys a batch
still uses.
"""
import ctypes as C
import json
import os
import re
import subprocess
import sys
import textwrap
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import pir_b200 as pb
from oracle import binding as ob
from oracle import client as oc
from tests.test_expansion_gpu import ROWS, _level_nodes, _limbs, _predicted_kernels, _row

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_POOL = ThreadPoolExecutor(max_workers=max(1, min(32, os.cpu_count() or 1)))  # the oracle's ctypes calls drop the GIL


# ------------------------------------------------------------------------------------------------ real clients
ITEM = 4096  # bytes per item: two per plaintext at N = 4096, four at 8192 (the trees have several levels)


class _Db:
    """A string database of n_items random items and the server over it."""

    def __init__(self, n, d, n_items, monkeypatch=None, tc=False):
        ep = pb.GenerateEncryptionParams(n, 20)
        self.p = pb.CreatePIRParameters(n_items, ITEM, d, ep)
        self.hp = oc.PIRParameters(self.p.num_items, self.p.num_pt, list(self.p.dimensions), self.p.bytes_per_item,
                                   self.p.items_per_plaintext, self.p.bits_per_coeff, n, ep.plain_modulus,
                                   list(ep.coeff_modulus))
        rng = np.random.default_rng(n_items * 31 + d)
        self.items = [rng.integers(0, 256, ITEM, dtype=np.uint8).tobytes() for _ in range(n_items)]
        if tc:  # the tensor-core scan takes batches of 4+ queries on any database size
            monkeypatch.setenv("PIRB_TC_MIN_PT", "0")
        self.db = pb.PIRDatabase.Create(self.items, self.p)
        if tc:
            monkeypatch.delenv("PIRB_TC_MIN_PT")
        self.server = pb.PIRServer.Create(self.db, self.p)
        self._ntt = None

    def clients(self, count, seed0=100):
        out = []
        for i in range(count):
            cl = oc.HarnessClient(self.hp, seed=seed0 + i)
            cl.gk = pb.GaloisKeys(cl.elts, cl.galois)
            out.append(cl)
        return out

    def db_ntt(self, orc):
        if self._ntt is None:
            self._ntt = oc.db_to_ntt(orc, oc.encode_string_db(self.hp, self.items))
        return self._ntt

    def requests(self, clients, order, sizes, seed):
        """One request per entry of `order` (client index), sizes[i] queries each; returns requests and indexes."""
        rng = np.random.default_rng(seed)
        reqs, idx = [], []
        for ci, nq in zip(order, sizes):
            want = [int(x) for x in rng.integers(0, self.p.num_items, nq)]
            reqs.append(pb.Request([clients[ci].create_query(i) for i in want], clients[ci].gk))
            idx.append(want)
        return reqs, idx

    def check(self, clients, order, reqs, idx, got, oracle=True):
        """Every response: ProcessRequest alone, the oracle with that client's keys, and the decrypted items."""
        assert len(got) == len(reqs)
        jobs = []
        for r, (req, resp) in enumerate(zip(reqs, got)):
            alone = self.server.ProcessRequest(req).reply
            assert len(resp.reply) == len(req.query) == len(alone)
            for i in range(len(alone)):
                assert np.array_equal(resp.reply[i], alone[i]), "request %d query %d differs from ProcessRequest" % (r, i)
            cl = clients[order[r]]
            assert cl.process_response_strings(idx[r], resp.reply) == [self.items[i] for i in idx[r]], r
            if oracle:
                ntt = self.db_ntt(cl.orc)
                for i, q in enumerate(req.query):
                    jobs.append((cl, ntt, q, resp.reply[i], "request %d query %d" % (r, i)))

        def one(job):
            cl, ntt, q, reply, tag = job
            want = cl.orc.process_query(ntt, self.p.dimensions, cl.elts, cl.galois, q)
            return None if np.array_equal(reply, want) else tag + ": differs from the oracle"

        errs = [e for e in _POOL.map(one, jobs) if e]
        assert not errs, errs[:8]


# (N, d, items, tensor-core scan, client order, queries per request): totals of 3 (CUDA-core batch scan), 8 and 20
MIX = {
    "n4096-d1-q3-permuted": (4096, 1, 40, False, [2, 0, 1], [1, 1, 1]),
    "n4096-d2-q8-ABA": (4096, 2, 60, True, [0, 1, 0, 2], [2, 3, 1, 2]),
    "n4096-d3-q20-repeats": (4096, 3, 60, True, [3, 1, 0, 1, 2, 4, 0, 3, 5], [3, 2, 3, 1, 2, 3, 2, 2, 2]),
    "n8192-d2-q3-ABA": (8192, 2, 30, False, [0, 1, 0], [1, 1, 1]),
    "n8192-d1-q8-permuted": (8192, 1, 30, True, [1, 2, 0, 1], [2, 2, 3, 1]),
}


@pytest.mark.parametrize("case", list(MIX))
def test_process_requests_matches_single_requests_oracle_and_items(case, monkeypatch):
    n, d, n_items, tc, order, sizes = MIX[case]
    h = _Db(n, d, n_items, monkeypatch, tc)
    clients = h.clients(max(order) + 1)
    reqs, idx = h.requests(clients, order, sizes, seed=len(order))
    h.check(clients, order, reqs, idx, h.server.ProcessRequests(reqs))


@pytest.mark.parametrize("n", [4096, 8192])
def test_one_client_is_byte_identical_to_pirb_answer(n, monkeypatch):
    """Requests all from one client: the batch equals pirb_answer of all their queries with that client's key."""
    h = _Db(n, 2, 30, monkeypatch, tc=True)
    clients = h.clients(1)
    reqs, idx = h.requests(clients, [0, 0, 0], [2, 3, 3], seed=5)
    got = h.server.ProcessRequests(reqs)
    whole = h.server.ProcessRequest(pb.Request([q for r in reqs for q in r.query], clients[0].gk)).reply
    flat = [x for resp in got for x in resp.reply]
    assert len(flat) == len(whole) == 8
    for a, b in zip(flat, whole):
        assert np.array_equal(a, b)
    assert clients[0].process_response_strings(idx[0], got[0].reply) == [h.items[i] for i in idx[0]]


@pytest.mark.parametrize("graphs", ["1", "0"])
def test_graph_lifecycle_serves_every_client_mix(graphs, monkeypatch):
    """Five calls of one shape (6 queries) with a different mix of clients each time: eager, capture, replays.  One
    graph per shape serves every mix because the key table is data.  PIRB_GRAPHS=0: the same calls run eagerly."""
    monkeypatch.setenv("PIRB_GRAPHS", graphs)
    h = _Db(4096, 2, 60, monkeypatch, tc=True)
    monkeypatch.delenv("PIRB_GRAPHS")
    clients = h.clients(4)
    mixes = [[0, 1, 2], [3, 3, 0], [2, 0, 1], [1, 3, 3], [0, 0, 0]]
    for call, order in enumerate(mixes):
        reqs, idx = h.requests(clients, order, [2, 2, 2], seed=100 + call)
        h.check(clients, order, reqs, idx, h.server.ProcessRequests(reqs), oracle=(call % 2 == 0))


def test_key_cache_smaller_than_the_batch():
    """20 clients in one call, key cache of 16: no handle of the batch may be closed before the call returns."""
    h = _Db(4096, 2, 40)
    clients = h.clients(20, seed0=500)
    assert h.server.key_cache_capacity == 16
    order = list(range(20))
    reqs, idx = h.requests(clients, order, [1] * 20, seed=20)
    h.check(clients, order, reqs, idx, h.server.ProcessRequests(reqs), oracle=False)
    assert len(h.server._multi_key_cache) == 16
    # and again in another order: 4 misses, 16 hits
    order = order[::-1]
    reqs = [reqs[i] for i in order]
    idx = [idx[i] for i in order]
    h.check(clients, list(range(20))[::-1], reqs, idx, h.server.ProcessRequests(reqs), oracle=False)


# ------------------------------------------------------------------------------------------------ the C ABI
def _table(handles):
    return (C.c_void_p * len(handles))(*[h.h.value if h is not None else None for h in handles])


def test_rejected_batches_launch_nothing_and_the_next_call_succeeds(monkeypatch):
    """A null handle, a handle without one level's Galois element (mid-batch) and a handle loaded on a context of other
    moduli are rejected with their status before anything runs: the reply buffer keeps its content.  A correct call
    follows each rejection."""
    from pir_b200 import _lib
    from pir_b200.api import _KeyHandle
    h = _Db(4096, 2, 40, monkeypatch, tc=True)
    ctx, L = h.server.ctx, _lib.lib()
    clients = h.clients(3)
    handles = [_KeyHandle(ctx, cl.gk) for cl in clients]
    reqs, idx = h.requests(clients, [0, 1, 2, 0], [1, 1, 1, 1], seed=9)
    q = np.ascontiguousarray(np.stack([r.query[0] for r in reqs]))
    want = [h.server.ProcessRequest(r).reply[0] for r in reqs]

    def call(tab):
        out = np.full((4, ctx.reply_cts, 2, ctx.k, ctx.N), 0xABCD, dtype=np.uint64)
        rc = L.pirb_answer_multi(ctx.h, tab, C.c_void_p(q.ctypes.data), 4, ctx.query_cts, C.c_void_p(out.ctypes.data))
        return rc, out

    def good():
        rc, out = call(_table([handles[0], handles[1], handles[2], handles[0]]))
        assert rc == 0, _lib.last_error()
        for i in range(4):
            assert np.array_equal(out[i], want[i]), i

    good()
    rc, out = call(_table([handles[0], None, handles[2], handles[0]]))
    assert rc == pb.INVALID_ARGUMENT and "query 1" in _lib.last_error()
    assert (out == 0xABCD).all()
    good()
    cl = clients[1]
    missing = cl.elts[0]  # N + 1: the first level of every tree
    keep = [i for i, e in enumerate(cl.elts) if e != missing]
    per = ctx.key_limbs
    lacking = _KeyHandle(ctx, pb.GaloisKeys([cl.elts[i] for i in keep],
                                            np.concatenate([cl.galois[i * per:(i + 1) * per] for i in keep])))
    rc, out = call(_table([handles[0], handles[1], lacking, handles[0]]))
    assert rc == pb.INTERNAL
    assert "Galois key not present for element %d" % missing in _lib.last_error() and "query 2" in _lib.last_error()
    assert (out == 0xABCD).all()
    good()
    other = _Db(4096, 2, 10, monkeypatch=None)
    ep2 = pb.EncryptionParameters(4096, ob.plain_modulus_batching(4096, 20), [int(x) for x in ROWS["q44k1-n4096"][1]()])
    p2 = pb.PIRParameters(num_items=1, num_pt=1, dimensions=[1], encryption_parameters=ep2, bytes_per_item=0,
                          items_per_plaintext=1, bits_per_coeff=0)
    db2 = pb.PIRDatabase(p2)
    elts = pb.generate_galois_elts(4096)
    foreign = _KeyHandle(db2.ctx, pb.GaloisKeys(elts, np.zeros(len(elts) * db2.ctx.key_limbs, dtype=np.uint64)))
    assert db2.ctx.key_limbs != ctx.key_limbs
    rc, out = call(_table([handles[0], handles[1], handles[2], foreign]))
    assert rc == pb.INVALID_ARGUMENT and "query 3" in _lib.last_error()
    assert (out == 0xABCD).all()
    good()
    del other


def test_multi_dev_on_one_stream_interleaved_with_answer_dev_on_another(monkeypatch):
    """pirb_answer_multi_dev on one torch stream and pirb_answer_dev on another, interleaved: the calls share the
    context's workspaces and key table, so each must wait for the previous one whatever its stream."""
    import torch
    from pir_b200 import _lib
    from pir_b200.api import _KeyHandle
    from pir_b200.sharded import _dp
    h = _Db(4096, 2, 60, monkeypatch, tc=True)
    ctx, L = h.server.ctx, _lib.lib()
    clients = h.clients(3)
    handles = [_KeyHandle(ctx, cl.gk) for cl in clients]
    order = [0, 1, 2, 1, 0, 2]
    reqs, idx = h.requests(clients, order, [1] * 6, seed=77)
    q = np.ascontiguousarray(np.stack([r.query[0] for r in reqs]))
    want = [h.server.ProcessRequest(r).reply[0] for r in reqs]
    d_q = torch.from_numpy(q.view(np.int64)).cuda()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    tab = _table([handles[i] for i in order])
    outs_multi, outs_one = [], []
    torch.cuda.synchronize()
    for it in range(4):
        om = torch.empty((6, ctx.reply_cts, 2, ctx.k, ctx.N), dtype=torch.int64, device="cuda")
        oo = torch.empty((2, ctx.reply_cts, 2, ctx.k, ctx.N), dtype=torch.int64, device="cuda")
        with torch.cuda.stream(s1):
            assert L.pirb_answer_multi_dev(ctx.h, tab, _dp(d_q), 6, ctx.query_cts, _dp(om),
                                           C.c_void_p(s1.cuda_stream)) == 0, _lib.last_error()
        with torch.cuda.stream(s2):  # queries 0 and 4 are client 0's
            d_q0 = d_q[[0, 4]].contiguous()
            assert L.pirb_answer_dev(ctx.h, handles[0].h, _dp(d_q0), 2, ctx.query_cts, _dp(oo),
                                     C.c_void_p(s2.cuda_stream)) == 0, _lib.last_error()
        outs_multi.append(om)
        outs_one.append(oo)
    torch.cuda.synchronize()
    for it in range(4):
        got = outs_multi[it].cpu().numpy().view(np.uint64)
        for i in range(6):
            assert np.array_equal(got[i], want[i]), (it, i)
        one = outs_one[it].cpu().numpy().view(np.uint64)
        assert np.array_equal(one[0], want[0]) and np.array_equal(one[1], want[4]), it
    ntt = h.db_ntt(clients[1].orc)
    assert np.array_equal(want[1], clients[1].orc.process_query(ntt, h.p.dimensions, clients[1].elts,
                                                                clients[1].galois, q[1]))


# ------------------------------------------------------------------------------------------------ every kernel
# rows of test_expansion_gpu chosen by the key-switch kernels they reach with 4 queries x 128 items (levels of 4..256
# nodes: the widest level takes the second generation for k <= 2)
KS_ROWS = ["n4096", "q44k1-n4096", "q44-n2048", "q44k1-n2048", "n8192", "q49-n4096", "q44-n4096-forced",
           "q30k8-n4096"]
KS_ITEMS = 128


def _ks_case(row):
    """Row parameters, a d = 1 database of KS_ITEMS plaintexts, two clients' random keys and four random queries."""
    n, mods, forced = _row(row)
    k = len(mods) - 1
    ep = pb.EncryptionParameters(n, ob.plain_modulus_batching(n, 20), mods)
    p = pb.PIRParameters(num_items=KS_ITEMS, num_pt=KS_ITEMS, dimensions=[KS_ITEMS], encryption_parameters=ep,
                         bytes_per_item=0, items_per_plaintext=1, bits_per_coeff=0)
    gks = []
    for seed in (1, 2):
        rng = np.random.default_rng(seed)
        elts = pb.generate_galois_elts(n)
        keys = np.stack([_limbs("uniform", q, (len(elts), k, 2, n), rng) for q in mods], axis=3)
        gks.append(pb.GaloisKeys(elts, np.ascontiguousarray(keys).reshape(-1)))
    rng = np.random.default_rng(3)
    qs = [np.ascontiguousarray(np.stack([_limbs("uniform", mods[j], (1, 2, n), rng) for j in range(k)], axis=2))
          for _ in range(4)]
    return n, mods, forced, p, gks, qs


def _ks_trace(row, out_dir):
    """One ProcessRequests call of the row (clients A, B, A, B) under torch.profiler: writes the key-switch kernels of
    the trace, the number of device events in it, the replies and the database (NTT form) to out_dir."""
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    n, mods, forced, p, gks, qs = _ks_case(row)
    if forced:
        os.environ["PIRB_KS_CLUSTER"] = "0"  # read at context creation
    db = pb.PIRDatabase(p)
    os.environ.pop("PIRB_KS_CLUSTER", None)
    db.fill_random(11)
    server = pb.PIRServer.Create(db, p)
    reqs = [pb.Request([qs[i]], gks[i % 2]) for i in range(4)]
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        got = server.ProcessRequests(reqs)
        torch.cuda.synchronize()
    names, events = set(), 0
    for ev in prof.events():
        events += ev.device_type == DeviceType.CUDA
        m = re.search(r"(k_ks_\w+)(<[^>]*>)?", ev.name)
        if m:
            names.add(m.group(1) + (m.group(2) or "").replace(" ", ""))
    with open(os.path.join(out_dir, row + ".json"), "w") as f:
        json.dump({"kernels": sorted(names), "device_events": events}, f)
    np.save(os.path.join(out_dir, row + "-replies.npy"), np.stack([g.reply[0] for g in got]))
    np.save(os.path.join(out_dir, row + "-db.npy"), db.read_ntt(0, KS_ITEMS))


_KS_SCRIPT = textwrap.dedent("""
    import sys
    sys.path.insert(0, sys.argv[1])
    from tests import test_multi_client_gpu as t
    for row in sys.argv[3:]:
        t._ks_trace(row, sys.argv[2])
    print("traced", len(sys.argv) - 3)
""")


@pytest.fixture(scope="module")
def ks_traces(tmp_path_factory):
    """The traces of every KS_ROWS row, taken in one fresh interpreter.  In a process that has been serving and
    profiling for minutes (a full suite), traces of one short call were seen to keep only its last few device events,
    so which kernels ran is read from a young process, as test_expansion_gpu reads its set-up order."""
    out = str(tmp_path_factory.mktemp("ks_traces"))
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", _KS_SCRIPT, ROOT, out] + KS_ROWS
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1200, cwd=ROOT)
    assert r.returncode == 0 and "traced %d" % len(KS_ROWS) in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]
    return out


@pytest.mark.parametrize("row", KS_ROWS)
def test_every_key_switch_kernel_picks_each_querys_key(row, ks_traces):
    """Random ring elements and random keys of two clients in the order A, B, A, B (adjacent queries differ, so a
    wrong query index in a kernel shows): every reply equals the oracle's with that query's keys, and the torch.profiler
    trace of the call shows that the predicted key-switch kernels ran."""
    import torch
    n, mods, forced, p, gks, qs = _ks_case(row)
    with open(os.path.join(ks_traces, row + ".json")) as f:
        trace = json.load(f)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    want = _predicted_kernels(n, mods, forced, _level_nodes(n, KS_ITEMS, 4), sms)
    assert set(trace["kernels"]) == want, (trace, sorted(want))
    got = np.load(os.path.join(ks_traces, row + "-replies.npy"))
    ntt = np.load(os.path.join(ks_traces, row + "-db.npy"))
    orc = ob.Oracle(n, mods, p.encryption_parameters.plain_modulus)

    def one(i):
        w = orc.process_query(ntt, p.dimensions, gks[i % 2].elts, gks[i % 2].data, qs[i])
        return None if np.array_equal(got[i], w) else "query %d differs from the oracle" % i

    errs = [e for e in _POOL.map(one, range(4)) if e]
    assert not errs, errs


# ------------------------------------------------------------------------------------------------ C++ host
def test_cpp_process_requests():
    """tests/cpp/multi_client_test.cpp (build/multi_client_test, built by `make all`)."""
    exe = os.path.join(ROOT, "build", "multi_client_test")
    assert os.path.exists(exe), "build/multi_client_test missing: run `make all`"
    r = subprocess.run([exe], capture_output=True, text=True, timeout=1200, cwd=ROOT)
    assert r.returncode == 0 and "ALL OK" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
