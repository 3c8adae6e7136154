"""The batched last-dimension scan on the tensor cores (pir_b200/csrc/kernels_tc.cu) across its launch geometry.

Every batch of 4 or more queries on a shard of 1024 or more plaintexts runs its last-dimension scan there (the
tensor-core scan, "TC scan" below).  Its host plan depends on the shape: byte limbs per residue (nb 5 up to 40-bit
moduli, 6 up to 48), dimL padded to 16 (Kp) and cut into 128-byte K chunks (kch), queries per MMA tile (qt 8 / 16 / 24)
and query tiles (n_qt), one or two shared-memory B buffers, 128-lane row tiles of 25 (nb 5) or 21 (nb 6) rows.  The
tests here choose shapes that reach each of these branches with small databases (explicit dimensions: a large dimL
with few rows), and compare the whole batch limb for limb with the CUDA-core batch scan on the same shard (a second
context with PIRB_TC_MIN=0, itself pinned to the oracle by test_gpu_parity.py), plus sampled (query, row) pairs with the
oracle's scan_row.  The plan itself (pir_b200/csrc/tc_plan.h) is checked for every shape on the CPU
(tests/cpp/device_math_host_test.cpp); the multi-GPU exchange and the ciphertext-multiplication mode on this path are
covered by rows of test_gpu_parity.py's parametrized tests.
"""
import numpy as np
import pytest

import pir_b200 as pb
from oracle import binding as ob

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------ helpers
def _find_ntt_primes(bits, n, count):
    out, v = [], (1 << bits) - 2 * n + 1
    while len(out) < count:
        if ob.is_prime(v):
            out.append(v)
        v -= 2 * n
    return out


def _encryption(mods):
    """n4096 / n8192: the default moduli of N=4096 (36-bit, nb 5) and N=8192 (43/44-bit, nb 6); q40 / q48: custom
    40-bit and 48-bit moduli at N=4096, the top of each byte width."""
    if mods == "n4096":
        return pb.GenerateEncryptionParams(4096, 20)
    if mods == "n8192":
        return pb.GenerateEncryptionParams(8192, 20)
    bits = {"q40": 40, "q48": 48}[mods]
    return pb.EncryptionParameters(4096, ob.plain_modulus_batching(4096, 20), _find_ntt_primes(bits, 4096, 3))


def _nb(ep):
    return (max(int(q).bit_length() for q in ep.coeff_modulus[:-1]) + 7) // 8


def _params(ep, rows, dimL):
    """dims [rows, dimL]; the last row is short unless dimL == 1."""
    short = dimL if dimL == 1 else max(1, (2 * dimL) // 3)
    num_pt = (rows - 1) * dimL + short
    return pb.PIRParameters(num_items=num_pt, num_pt=num_pt, dimensions=[rows, dimL], encryption_parameters=ep,
                            bytes_per_item=0, items_per_plaintext=1, bits_per_coeff=0)


def _residues(fill, q, shape, rng, nb):
    """Host residues mod q: uniform; all q-1; or a random top limb over all-0xFF lower limbs (every byte product of
    the lower limbs is 255^2 and the limb recombination carries as far as it can)."""
    if fill == "random":
        return rng.integers(0, q, shape, dtype=np.uint64)
    if fill == "qminus1":
        return np.full(shape, q - 1, dtype=np.uint64)
    s = 8 * (nb - 1)
    hi = rng.integers(0, q >> s, shape, dtype=np.uint64)
    return (hi << np.uint64(s)) | np.uint64((1 << s) - 1)


def _device_residues(torch, fill, q, shape, gen, nb):
    """_residues on the device (the selection vectors of a large dimL are gigabytes)."""
    if fill == "random":
        return torch.randint(0, q, shape, generator=gen, device="cuda", dtype=torch.int64)
    if fill == "qminus1":
        return torch.full(shape, q - 1, device="cuda", dtype=torch.int64)
    s = 8 * (nb - 1)
    hi = torch.randint(0, q >> s, shape, generator=gen, device="cuda", dtype=torch.int64)
    return (hi << s) | ((1 << s) - 1)


def _shards(p, fill, seed, monkeypatch):
    """(tensor-core context, CUDA-core context) over the same database content.  The tensor-core one takes every batch
    of >= 4 queries whatever the shard size (PIRB_TC_MIN_PT=0); the other never uses the tensor cores (PIRB_TC_MIN=0)."""
    from pir_b200 import sharded
    monkeypatch.setenv("PIRB_TC_MIN_PT", "0")
    tc = sharded.ShardServer(p, device=0)
    monkeypatch.delenv("PIRB_TC_MIN_PT")
    monkeypatch.setenv("PIRB_TC_MIN", "0")
    ref = sharded.ShardServer(p, device=0)
    monkeypatch.delenv("PIRB_TC_MIN")
    if fill == "random":
        tc.db.fill_random(seed)
        ref.db.fill_random(seed)
    else:
        ep = p.encryption_parameters
        rng = np.random.default_rng(seed)
        k, n = len(ep.coeff_modulus) - 1, ep.poly_modulus_degree
        limbs = np.stack([_residues(fill, int(ep.coeff_modulus[j]), (p.num_pt, n), rng, _nb(ep)) for j in range(k)],
                         axis=1)
        tc.db.load_ntt(limbs)
        ref.db.load_ntt(limbs)
    return tc, ref


def _selection_vectors(p, nq, fill, seed):
    """[nq][dimL][2][k][N] NTT-form selection entries on the device."""
    import torch
    ep = p.encryption_parameters
    k, n, dimL = len(ep.coeff_modulus) - 1, ep.poly_modulus_degree, p.dimensions[-1]
    gen = torch.Generator(device="cuda")
    gen.manual_seed(seed)
    sv = torch.empty((nq, dimL, 2, k, n), dtype=torch.int64, device="cuda")
    for j in range(k):
        sv[:, :, :, j, :] = _device_residues(torch, fill, int(ep.coeff_modulus[j]), (nq, dimL, 2, n), gen, _nb(ep))
    return sv


def _sampled_queries(nq):
    """The first and last query, and the first query of every query tile after the first (tiles are 8, 16 or 24
    queries, so every multiple of 8 is the start of some tile)."""
    return sorted({0, nq - 1} | set(range(8, nq, 8)))


def _check_scan(p, nq, fill, monkeypatch, qt_env=None, seed=1):
    import torch
    tc, ref = _shards(p, fill, seed, monkeypatch)
    sv = _selection_vectors(p, nq, fill, seed + 1)
    if qt_env is not None:
        monkeypatch.setenv("PIRB_TC_QT", qt_env)
    got = tc.scan(sv)
    if qt_env is not None:
        monkeypatch.delenv("PIRB_TC_QT")
    want = ref.scan(sv)
    torch.cuda.synchronize()
    n_rows = got.shape[1]
    assert got.shape == want.shape == (nq, n_rows, 2, tc.k, tc.N)
    if not torch.equal(got, want):
        bad = (got != want).nonzero()
        pytest.fail("tensor-core scan differs from the CUDA-core scan at %d limbs, first (query, row, poly, modulus, "
                    "coefficient) %s" % (bad.shape[0], tuple(bad[0].tolist())))
    ep = p.encryption_parameters
    orc = ob.Oracle(ep.poly_modulus_degree, list(ep.coeff_modulus), ep.plain_modulus)
    dimL = p.dimensions[-1]
    got_h = got.cpu().numpy().view(np.uint64)
    for i in _sampled_queries(nq):
        sv_i = sv[i].cpu().numpy().view(np.uint64)
        for r in sorted({0, n_rows // 2, n_rows - 1}):
            first = r * dimL
            cnt = min(dimL, p.num_pt - first)
            want_row = orc.scan_row(tc.db.read_ntt(first, cnt), sv_i[:cnt])
            assert np.array_equal(got_h[i, r], want_row), (i, r)
    del got, want, sv
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ geometry matrix
# (moduli, dimL, rows, queries, PIRB_TC_QT, fill).  rpt = 25 rows per tile for nb 5, 21 for nb 6; the default qt is 16.
MATRIX = [
    # nb 5, default N=4096 moduli
    ("n4096", 1, 53, 4, None, "random"),        # dimL 1: Kp 16, one partial K chunk; 2*rpt + 3 rows, every row full
    ("n4096", 16, 24, 8, None, "random"),       # rpt - 1 rows: one tile, last lane group idle
    ("n4096", 17, 25, 9, None, "random"),       # rpt rows; 9 queries: qt 16 with 7 padded query columns
    ("n4096", 128, 26, 16, None, "random"),     # rpt + 1 rows: a second tile holding one short row; Kp 128, kch 1
    ("n4096", 129, 53, 17, None, "random"),     # kch 2 with a 16-byte last chunk; n_qt 2
    ("n4096", 300, 1, 24, None, "random"),      # one short row; n_qt 2, second tile half padding
    ("n4096", 300, 3, 33, None, "random"),      # n_qt 3; b_bufs 2 at kch 3
    ("n4096", 385, 3, 16, None, "random"),      # Kp 400 (Kp % 128 == 16), kch 4: b_bufs 1
    ("n4096", 640, 2, 9, None, "random"),       # kch 5
    ("n4096", 664, 2, 16, None, "random"),      # configs[4] d=2 last dimension: kch 6, Kp % 128 == 32
    ("n4096", 1024, 2, 16, None, "random"),     # kch 8 (Kp % 128 == 0): the widest B operand of qt 16
    ("n4096", 1024, 2, 4, None, "random"),      # qt 8
    ("n4096", 128, 3, 17, "8", "random"),       # qt 8: n_qt 3
    ("n4096", 385, 2, 9, "8", "random"),        # qt 8, kch 4, b_bufs 2
    ("n4096", 300, 2, 24, "24", "random"),      # qt 24: N of the MMA = 240, one tile
    ("n4096", 129, 26, 33, "24", "random"),     # qt 24, n_qt 2, second tile 15 padded queries
    ("n4096", 640, 2, 24, "24", "random"),      # qt 24 at its widest fitting K: b_bufs 1
    # nb 6, default N=8192 moduli
    ("n8192", 1, 21, 4, None, "random"),
    ("n8192", 17, 20, 4, None, "random"),       # rpt - 1 rows
    ("n8192", 128, 21, 9, None, "random"),      # rpt rows, qt 16 (N of the MMA = 192)
    ("n8192", 129, 22, 16, None, "random"),     # rpt + 1 rows
    ("n8192", 16, 45, 17, None, "random"),      # 2*rpt + 3 rows, n_qt 2
    ("n8192", 300, 2, 16, None, "random"),      # b_bufs 1 (nb 6, qt 16, dimL >= 257)
    ("n8192", 640, 2, 16, None, "random"),      # kch 5: the widest B operand of nb 6 at qt 16
    ("n8192", 664, 2, 8, None, "random"),       # qt 8, kch 6, b_bufs 1
    ("n8192", 129, 2, 24, "8", "random"),       # qt 8, n_qt 3
    ("n8192", 129, 2, 33, None, "random"),      # n_qt 3 at nb 6
    # top of each byte width
    ("q40", 385, 25, 9, None, "random"),
    ("q40", 17, 53, 33, None, "random"),
    ("q48", 129, 22, 17, None, "random"),
    ("q48", 640, 2, 16, None, "random"),
    # limb recombination and the 128-bit carries at their maximum
    ("q48", 1024, 2, 8, None, "qminus1"),
    ("q40", 1024, 2, 16, None, "qminus1"),
    ("n4096", 1024, 2, 16, None, "ff"),
    ("n8192", 640, 2, 16, None, "ff"),
    ("q48", 300, 26, 9, None, "ff"),
    # B operands too wide for the requested query tile: the plan narrows the tile
    ("n8192", 700, 2, 9, None, "random"),       # nb 6, dimL > 640: qt 8, n_qt 2
    ("q48", 1024, 2, 9, None, "random"),        # nb 6 at the top of its width: qt 8, n_qt 2
    ("n4096", 700, 2, 24, "24", "random"),      # qt 24 requested, qt 16 fits: n_qt 2
    ("n4096", 2048, 2, 4, None, "random"),      # kch 16, the widest nb 5 operand: b_bufs 1, two A stages
    ("n8192", 1280, 2, 4, None, "random"),      # kch 10, the widest nb 6 operand: b_bufs 1, two A stages
]


def _case_id(c):
    mods, dimL, rows, nq, qt, fill = c
    return "%s-L%d-r%d-q%d%s-%s" % (mods, dimL, rows, nq, "" if qt is None else "-qt" + qt, fill)


@pytest.mark.parametrize("case", MATRIX, ids=_case_id)
def test_tc_scan_geometry_matches_cuda_core_scan_and_oracle(case, monkeypatch):
    """ShardServer.scan (pirb_scan_dev, never graphed) on the tensor cores against the CUDA-core batch scan of the same
    shard, limb for limb, and sampled (query, row) pairs against the oracle: the first and last query and the first
    query of every later query tile, the first, a middle and the short last row."""
    mods, dimL, rows, nq, qt_env, fill = case
    _check_scan(_params(_encryption(mods), rows, dimL), nq, fill, monkeypatch, qt_env)


# ------------------------------------------------------------------------------------------------ large B operands
# Shapes whose B operand at the requested query tile does not fit shared memory: dims [2, 1100] at N=4096 with 9 and
# 16 queries (nb 5, qt 16, kch 9), dims [2, 700] at N=8192 with 9 queries (nb 6, qt 16, kch 6), dims [2, 700] at N=4096
# with qt 24 — all scanned with a narrower query tile — and dims [2, 2100] at N=4096 (kch 17: no query tile fits, the
# batch is scanned on the CUDA cores).
LARGE = [("n4096", 1100, 9, None), ("n4096", 1100, 16, None), ("n8192", 700, 9, None), ("n4096", 700, 24, "24"),
         ("n4096", 2100, 4, None)]


def _large_id(c):
    mods, dimL, nq, qt = c
    return "%s-L%d-q%d%s" % (mods, dimL, nq, "" if qt is None else "-qt" + qt)


@pytest.mark.parametrize("case", LARGE, ids=_large_id)
def test_large_last_dimension_scan_matches_cuda_core_scan_and_oracle(case, monkeypatch):
    mods, dimL, nq, qt_env = case
    _check_scan(_params(_encryption(mods), 2, dimL), nq, "random", monkeypatch, qt_env)


@pytest.mark.parametrize("case", LARGE, ids=_large_id)
def test_large_last_dimension_process_request_matches_oracle(case, monkeypatch):
    """The same shapes end to end: PIRServer.ProcessRequest of the whole batch (a shard of >= 1024 plaintexts, so the
    default thresholds apply), sampled queries against the oracle's ProcessRequest on the whole database."""
    mods, dimL, nq, qt_env = case
    if qt_env is not None:
        monkeypatch.setenv("PIRB_TC_QT", qt_env)
    ep = _encryption(mods)
    p = _params(ep, 2, dimL)
    n, mods_l = ep.poly_modulus_degree, [int(q) for q in ep.coeff_modulus]
    k = len(mods_l) - 1
    db = pb.PIRDatabase(p)
    db.fill_random(29)
    server = pb.PIRServer.Create(db, p)
    db_ntt = db.read_ntt(0, p.num_pt)
    rng = np.random.default_rng(dimL + nq)
    elts = [(n >> i) + 1 for i in range(n.bit_length() - 1)]
    keys = np.stack([rng.integers(0, q, (len(elts), k, 2, n), dtype=np.uint64) for q in mods_l], axis=3)
    gk = pb.GaloisKeys(elts, keys.reshape(-1))
    n_ct = server.ctx.query_cts
    queries = np.stack([rng.integers(0, q, (nq, n_ct, 2, n), dtype=np.uint64) for q in mods_l[:k]], axis=3)
    got = server.ProcessRequest(pb.Request([q for q in queries], gk)).reply
    assert len(got) == nq
    orc = ob.Oracle(n, mods_l, ep.plain_modulus)
    for i in _sampled_queries(nq):
        want = orc.process_query(db_ntt, p.dimensions, elts, keys.reshape(-1), queries[i])
        assert np.array_equal(got[i], want), i


# ------------------------------------------------------------------------------------------------ database reloads
@pytest.mark.parametrize("graphs", [1, 0])
@pytest.mark.parametrize("reload", ["load_ntt", "fill_random"])
def test_batched_answers_follow_database_reloads(reload, graphs, monkeypatch):
    """The TC scan reads a byte-planar copy of the database, and repeated batches replay a captured graph of the answer
    path.  A database load between answers must reach both: three answers (eager, capture, replay), a reload of part
    (load_ntt) or all (fill_random under a new seed) of the database, two more answers — every reply equal to the
    oracle's on the database as it is at that moment.  graphs = 0 (PIRB_GRAPHS=0) is the eager control."""
    monkeypatch.setenv("PIRB_TC_MIN_PT", "0")
    if not graphs:
        monkeypatch.setenv("PIRB_GRAPHS", "0")
    n, nq = 4096, 5
    ep = pb.GenerateEncryptionParams(n, 20)
    p = pb.CreatePIRParameters(82, 0, 2, ep)
    assert p.dimensions == [10, 9]
    mods = [int(q) for q in ep.coeff_modulus]
    k = len(mods) - 1
    rng = np.random.default_rng(5 + graphs)
    orc = ob.Oracle(n, mods, ep.plain_modulus)
    coeffs = rng.integers(0, ep.plain_modulus, (p.num_pt, n), dtype=np.uint64)
    db = pb.PIRDatabase(p)
    db.load_coeff(coeffs)
    server = pb.PIRServer.Create(db, p)
    db_ntt = np.stack([orc.plain_to_ntt(c) for c in coeffs])
    elts = [(n >> i) + 1 for i in range(12)]
    keys = np.stack([rng.integers(0, q, (len(elts), k, 2, n), dtype=np.uint64) for q in mods], axis=3)
    gk = pb.GaloisKeys(elts, keys.reshape(-1))

    def answer_and_check(tag):
        queries = np.stack([rng.integers(0, q, (nq, 1, 2, n), dtype=np.uint64) for q in mods[:k]], axis=3)
        got = server.ProcessRequest(pb.Request([q for q in queries], gk)).reply
        for i in range(nq):
            want = orc.process_query(db_ntt, p.dimensions, elts, keys.reshape(-1), queries[i])
            assert np.array_equal(got[i], want), (tag, i)

    for call in range(3):
        answer_and_check(("before", call))
    if reload == "load_ntt":
        new = np.stack([rng.integers(0, q, (30, n), dtype=np.uint64) for q in mods[:k]], axis=1)
        db.load_ntt(new, 20)
        db_ntt[20:50] = new
    else:
        db.fill_random(1234)
        db_ntt = db.read_ntt(0, p.num_pt)
    for call in range(2):
        answer_and_check(("after", call))


def test_peer_exchange_flow_follows_database_reloads(monkeypatch):
    """pirb_dist_* is not graphed, but its consumers scan the byte-planar copy too: after a reload of part of the
    database the next step must rebuild it before its first scan.  Two ranks on this GPU, tensor-core exchange."""
    from pir_b200 import sharded
    monkeypatch.setenv("PIRB_TC_MIN_PT", "0")
    n, world, ql = 4096, 2, 5
    ep = pb.GenerateEncryptionParams(n, 20)
    p = pb.CreatePIRParameters(300, 0, 2, ep)
    mods = [int(q) for q in ep.coeff_modulus]
    k = len(mods) - 1
    rng = np.random.default_rng(41)
    orc = ob.Oracle(n, mods, ep.plain_modulus)
    grp = sharded.ShardGroup(p, [0] * world, ql, 2)
    coeffs = rng.integers(0, ep.plain_modulus, (p.num_pt, n), dtype=np.uint64)
    grp.load_coeff(coeffs)
    elts = [(n >> i) + 1 for i in range(12)]
    keys = np.stack([rng.integers(0, q, (len(elts), k, 2, n), dtype=np.uint64) for q in mods], axis=3)
    grp.set_keys(pb.GaloisKeys(elts, keys.reshape(-1)))
    n_ct = sum(p.dimensions) // n + 1
    for step in range(3):
        if step == 2:
            coeffs[100:250] = rng.integers(0, ep.plain_modulus, (150, n), dtype=np.uint64)
            grp.load_coeff(coeffs[100:250], 100)
        db_ntt = np.stack([orc.plain_to_ntt(c) for c in coeffs])
        queries = np.stack([rng.integers(0, q, (world, ql, n_ct, 2, n), dtype=np.uint64) for q in mods[:k]], axis=4)
        outs = grp.answer([sharded.to_device(queries[r], "cuda:0") for r in range(world)])
        for r in range(world):
            got = sharded.to_host(outs[r])
            for i in range(ql):
                want = orc.process_query(db_ntt, p.dimensions, elts, keys.reshape(-1), queries[r, i])
                assert np.array_equal(got[i], want), (step, r, i)
