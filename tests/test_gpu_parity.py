"""GPU parity tests (run with -m gpu on the B200 box): every C-ABI entry point of the answer path against the CPU
oracle on the same seeded inputs — bit-exact on all limbs — plus decrypt-level checks against the reference's
known-answer vectors and size-independent properties at BASELINE.json's sizes.
"""
import dataclasses
import json
import os

import numpy as np
import pytest

import pir_b200 as pb
from oracle import binding as ob
from oracle import client as oc

pytestmark = pytest.mark.gpu
N = 4096


def _params(dbsize, elem=0, d=1, n=4096, bits=20, bpc=0, ct_mult=False):
    ep = pb.GenerateEncryptionParams(n, bits)
    return pb.CreatePIRParameters(dbsize, elem, d, ep, ct_mult, bpc)


def _harness(p, seed=1):
    ep = p.encryption_parameters
    hp = oc.PIRParameters(p.num_items, p.num_pt, list(p.dimensions), p.bytes_per_item, p.items_per_plaintext,
                          p.bits_per_coeff, ep.poly_modulus_degree, ep.plain_modulus, list(ep.coeff_modulus),
                          bool(p.use_ciphertext_multiplication))
    return oc.HarnessClient(hp, seed=seed)


def _gk(cl, elts=None, seed=77):
    elts = cl.elts if elts is None else elts
    data = cl.galois if elts is cl.elts else cl.orc.galois_keys(cl.keys, elts, seed)
    return pb.GaloisKeys(elts, data), data


def _random_items(p, seed=42):
    rng = np.random.default_rng(seed)
    return [rng.integers(0, 256, p.bytes_per_item, dtype=np.uint8).tobytes() for _ in range(p.num_items)]


def _random_ct(orc, rng):
    return np.stack([rng.integers(0, orc.moduli[j], orc.N, dtype=np.uint64) for _ in range(2) for j in range(orc.k)]
                    ).reshape(2, orc.k, orc.N)


@pytest.fixture(scope="module")
def srv10():
    """server_test.cpp fixture: 10 items x 7680 B, N=4096, t 20 bit; integer database."""
    p = _params(10, 7680, 1)
    cl = _harness(p, seed=42)
    rng = np.random.default_rng(42)
    vals = [int(v) for v in rng.integers(0, 1 << 48, 10, dtype=np.int64)]
    db = pb.PIRDatabase.Create(vals, p)
    server = pb.PIRServer.Create(db, p)
    return p, cl, vals, db, server


# ------------------------------------------------------------------------------------------------
def test_db_preprocess_matches_oracle(srv10):
    p, cl, vals, db, server = srv10
    want = oc.db_to_ntt(cl.orc, oc.encode_int_db(cl.params, vals))
    assert np.array_equal(db.read_ntt(0, 10), want)


@pytest.mark.parametrize("n,bits", [(4096, 16), (8192, 20)])
def test_populate_strings_matches_oracle(n, bits):
    p = _params(23, 0, 1, n, bits)
    cl = _harness(p)
    items = _random_items(p)
    db = pb.PIRDatabase.Create(items, p)
    assert db.size() == p.num_pt
    want = oc.db_to_ntt(cl.orc, oc.encode_string_db(cl.params, items))
    assert np.array_equal(db.read_ntt(0, p.num_pt), want)
    with pytest.raises(pb.PIRStatusError) as e:  # database_test.cpp:326-339 / database.cpp:85-90
        pb.PIRDatabase.Create(items[:-1], p)
    assert e.value.code == pb.INVALID_ARGUMENT


# ------------------------------------------------------------------------------------------------ substitution
SUBST = [("42", 3, "42"), ("1x^1", 5, "1x^5"), ("6x^2", 3, "6x^6"), ("1x^1", N + 1, "FC000x^1"),
         ("1x^4", N + 1, "1x^4"), ("1x^8", N // 2 + 1, "1x^8"), ("1x^8", N // 4 + 1, "1x^8"),
         ("1x^8", N // 8 + 1, "FC000x^8"), ("77x^4095", 3, "77x^4093"), ("1x^4095", N + 1, "FC000x^4095"),
         ("4x^4 + 33x^3 + 222x^2 + 19x^1 + 42", N + 1, "4x^4 + FBFCEx^3 + 222x^2 + FBFE8x^1 + 42")]


@pytest.mark.parametrize("inp,power,expected", SUBST)
def test_substitute_kat_and_bit_exact(srv10, inp, power, expected):
    # server_test.cpp:271-305
    p, cl, vals, db, server = srv10
    ct = cl.encrypt(oc.parse_hex_poly(inp, N))
    gk, raw = _gk(cl, [power])
    want = cl.orc.substitute(ct, power, [power], raw)
    got = ct.copy()
    server.substitute_power_x_inplace(got, power, gk)
    assert np.array_equal(got, want)
    assert oc.format_hex_poly(cl.decrypt(got)) == oc.format_hex_poly(oc.parse_hex_poly(expected, N))


def test_substitute_missing_key(srv10):
    p, cl, vals, db, server = srv10
    gk, _ = _gk(cl, [5])
    ct = cl.encrypt(oc.parse_hex_poly("1x^1", N))
    with pytest.raises(pb.PIRStatusError) as e:
        server.substitute_power_x_inplace(ct, 3, gk)
    assert e.value.code == pb.INTERNAL  # server.cpp:72-74


def test_substitute_random_ciphertexts_all_levels(srv10):
    p, cl, vals, db, server = srv10
    rng = np.random.default_rng(3)
    gk, raw = _gk(cl)
    for g in cl.elts:
        ct = _random_ct(cl.orc, rng)
        want = cl.orc.substitute(ct, g, cl.elts, raw)
        got = ct.copy()
        server.substitute_power_x_inplace(got, g, gk)
        assert np.array_equal(got, want), g


# ------------------------------------------------------------------------------------------------ shifts
@pytest.mark.parametrize("inp,k,expected", [("42x^1", 1, "42"), ("42x^42", 41, "42x^1"),
                                            ("1x^4 + 1x^3 + 1x^1", 1, "1x^3 + 1x^2 + 1"),
                                            ("1x^16 + 1x^12 + 1x^8", 4, "1x^12 + 1x^8 + 1x^4")])
def test_multiply_inverse_power_x(srv10, inp, k, expected):
    # server_test.cpp:307-339
    p, cl, vals, db, server = srv10
    ct = cl.encrypt(oc.parse_hex_poly(inp, N))
    got = server.multiply_inverse_power_of_x(ct, k)
    assert np.array_equal(got, cl.orc.mul_inv_pow_x(ct, k))
    assert oc.format_hex_poly(cl.decrypt(got)) == oc.format_hex_poly(oc.parse_hex_poly(expected, N))


def test_multiply_inverse_power_x_all_ranges(srv10):
    p, cl, vals, db, server = srv10
    rng = np.random.default_rng(4)
    ct = _random_ct(cl.orc, rng)
    ct[0, 0, :7] = 0  # zeros stay zeros under negation
    for k in (0, 1, 2, 4095, 4096, 4097, N + 64, 2 * N - 1, 2 * N, 2 * N + 5):
        assert np.array_equal(server.multiply_inverse_power_of_x(ct, k), cl.orc.mul_inv_pow_x(ct, k)), k


# ------------------------------------------------------------------------------------------------ expansion
@pytest.mark.parametrize("inp,expected", [("1", ["2", "0"]), ("1x^1", ["0", "2"]),
                                          ("3x^3 + 2x^2 + 1x^1 + 42", ["108", "4", "8", "C"]),
                                          ("1x^5", ["0", "0", "0", "0", "0", "8"])])
def test_oblivious_expansion_kat(srv10, inp, expected):
    # server_test.cpp:341-383
    p, cl, vals, db, server = srv10
    ct = cl.encrypt(oc.parse_hex_poly(inp, N))
    gk, raw = _gk(cl)
    got = server.oblivious_expansion(ct, len(expected), gk)
    want = cl.orc.expand(ct, len(expected), cl.elts, raw, single=True)
    assert np.array_equal(got, want)
    for o, e in zip(got, expected):
        assert oc.format_hex_poly(cl.decrypt(o)) == oc.format_hex_poly(oc.parse_hex_poly(e, N))


@pytest.mark.parametrize("num_items", [1, 2, 3, 17, 100, 1000])
def test_oblivious_expansion_single_sizes(srv10, num_items):
    p, cl, vals, db, server = srv10
    rng = np.random.default_rng(num_items)
    ct = _random_ct(cl.orc, rng)
    gk, raw = _gk(cl)
    assert np.array_equal(server.oblivious_expansion(ct, num_items, gk),
                          cl.orc.expand(ct, num_items, cl.elts, raw, single=True))


@pytest.mark.parametrize("num_items,index,expected_value", [(100, 42, 128), (4096, 3007, 4096), (5000, 4095, 4096),
                                                            (5000, 4200, 1024)])
def test_oblivious_expansion_multi_ct(srv10, num_items, index, expected_value):
    # server_test.cpp:385-428
    p, cl, vals, db, server = srv10
    n_ct = num_items // N + 1
    cts = []
    for i in range(n_ct):
        pt = np.zeros(N, dtype=np.uint64)
        if index // N == i:
            pt[index % N] = 1
        cts.append(cl.encrypt(pt))
    cts = np.stack(cts)
    gk, raw = _gk(cl)
    got = server.oblivious_expansion(cts, num_items, gk)
    assert got.shape[0] == num_items
    want = cl.orc.expand(cts, num_items, cl.elts, raw)
    assert np.array_equal(got, want)
    for i in sorted({index, 0, num_items - 1}):
        pt = cl.decrypt(got[i])
        assert int(pt[0]) == (expected_value if i == index else 0) and not pt[1:].any()


def test_expansion_argument_errors(srv10):
    p, cl, vals, db, server = srv10
    gk, _ = _gk(cl)
    ct = cl.encrypt(np.zeros(N, dtype=np.uint64))
    with pytest.raises(pb.PIRStatusError) as e:  # server.cpp:111-114
        server.oblivious_expansion(ct, N + 1, gk)
    assert e.value.code == pb.INVALID_ARGUMENT
    with pytest.raises(pb.PIRStatusError) as e:  # server.cpp:154-158
        server.oblivious_expansion(np.stack([ct, ct]), 100, gk)
    assert e.value.code == pb.INVALID_ARGUMENT
    gk5, _ = _gk(cl, [5])
    with pytest.raises(pb.PIRStatusError) as e:  # missing key -> Internal
        server.oblivious_expansion(ct, 4, gk5)
    assert e.value.code == pb.INTERNAL


# ------------------------------------------------------------------------------------------------ PIRDatabase::multiply
def _selection_vector(cl, dims, indices):
    cts = []
    for d, dim in enumerate(dims):
        for i in range(dim):
            pt = np.zeros(cl.orc.N, dtype=np.uint64)
            if i == indices[d]:
                pt[0] = 1
            cts.append(cl.encrypt(pt))
    return np.stack(cts)


@pytest.mark.parametrize("n,bits,dbsize,d,idx", [(4096, 16, 10, 1, 7), (4096, 16, 16, 2, 11), (4096, 16, 16, 2, 0),
                                                  (4096, 16, 16, 2, 15), (4096, 16, 82, 2, 42), (8192, 20, 27, 3, 2),
                                                  (8192, 20, 117, 3, 17), (4096, 20, 200, 1, 199), (4096, 20, 50, 3, 49),
                                                  (4096, 24, 77, 4, 5)])
def test_multiply_multi_dim(n, bits, dbsize, d, idx):
    # database_test.cpp:343-388 (CTDecomp arm) + extra shapes; bit-exact vs the oracle and decrypt-correct
    p = _params(dbsize, 0, d, n, bits)
    cl = _harness(p, seed=11)
    items = _random_items(p)
    db = pb.PIRDatabase.Create(items, p)
    sv = _selection_vector(cl, p.dimensions, db.calculate_indices(idx))
    want, sv_after = cl.orc.db_multiply(oc.db_to_ntt(cl.orc, oc.encode_string_db(cl.params, items)), p.dimensions, sv)
    got_sv = sv.copy()
    got = db.multiply(got_sv)
    assert got.shape[0] == (2 * cl.orc.ER) ** (d - 1)
    assert np.array_equal(got, want)
    assert np.array_equal(got_sv, sv_after)  # in-place NTT of the selection vector (database.cpp:190,222)
    if d <= 3:
        res = cl.process_reply(got)
        assert ob.string_decode(res, cl.orc.ptb, p.bytes_per_item) == items[idx]


def test_multiply_integer_dot_product():
    # database_test.cpp:155-178
    p = _params(10, 0, 1)
    cl = _harness(p, seed=3)
    rng = np.random.default_rng(8)
    vals = [int(v) for v in rng.integers(0, 1 << 20, 10)]
    db = pb.PIRDatabase.Create(vals, p)
    v = list(range(-5, 5))
    sv = np.stack([cl.encrypt(oc.integer_encode(x, N, cl.orc.t)) for x in v])
    out = db.multiply(sv)
    assert oc.integer_decode(cl.decrypt(out[0]), cl.orc.t) == sum(a * b for a, b in zip(v, vals))


def test_multiply_selection_vector_size_errors():
    # database_test.cpp:180-219
    p = _params(100, 0, 2)
    db = pb.PIRDatabase.Create(p)
    k = len(p.encryption_parameters.coeff_modulus) - 1
    for n_sv in (19, 21):
        with pytest.raises(pb.PIRStatusError) as e:
            db.multiply(np.zeros((n_sv, 2, k, N), dtype=np.uint64))
        assert e.value.code == pb.INVALID_ARGUMENT


# ------------------------------------------------------------------------------------------------ ProcessRequest
def test_process_request_single_ct(srv10):
    # server_test.cpp:98-121
    p, cl, vals, db, server = srv10
    gk, raw = _gk(cl)
    pt = np.zeros(N, dtype=np.uint64); pt[7] = 1
    q = cl.encrypt(pt)[None]
    resp = server.ProcessRequest(pb.Request([q], gk))
    assert len(resp.reply) == 1 and resp.reply[0].shape[0] == 1
    want = cl.orc.process_query(db.read_ntt(0, 10), p.dimensions, cl.elts, raw, q)
    assert np.array_equal(resp.reply[0], want)
    assert oc.integer_decode(cl.decrypt(resp.reply[0][0]), cl.orc.t) == vals[7] * pb.next_power_two(10)


def test_process_request_multi_ct():
    # server_test.cpp:123-151
    p = _params(5000, 7680, 1)
    cl = _harness(p, seed=9)
    rng = np.random.default_rng(42)
    vals = [int(v) for v in rng.integers(0, 1 << 48, 5000, dtype=np.int64)]
    db = pb.PIRDatabase.Create(vals, p)
    server = pb.PIRServer.Create(db, p)
    gk, raw = _gk(cl)
    idx = 4200
    pt = np.zeros(N, dtype=np.uint64); pt[idx - N] = 1
    q = np.stack([cl.encrypt(np.zeros(N, dtype=np.uint64)), cl.encrypt(pt)])
    resp = server.ProcessRequest(pb.Request([q], gk))
    want = cl.orc.process_query(db.read_ntt(0, 5000), p.dimensions, cl.elts, raw, q)
    assert np.array_equal(resp.reply[0], want)
    assert oc.integer_decode(cl.decrypt(resp.reply[0][0]), cl.orc.t) == vals[idx] * pb.next_power_two(5000 - N)
    with pytest.raises(pb.PIRStatusError) as e:  # one ct short (server.cpp:154-158)
        server.ProcessRequest(pb.Request([q[:1]], gk))
    assert e.value.code == pb.INVALID_ARGUMENT


def test_process_request_batch_and_zero(srv10):
    # server_test.cpp:153-207
    p, cl, vals, db, server = srv10
    gk, raw = _gk(cl)
    qs = []
    for idx in (3, 4, 5):
        pt = np.zeros(N, dtype=np.uint64); pt[idx] = 1
        qs.append(cl.encrypt(pt)[None])
    qs.append(cl.encrypt(np.zeros(N, dtype=np.uint64))[None])
    resp = server.ProcessRequest(pb.Request(qs, gk))
    assert len(resp.reply) == 4
    dbn = db.read_ntt(0, 10)
    for q, r, exp in zip(qs, resp.reply, [vals[3] * 16, vals[4] * 16, vals[5] * 16, 0]):
        assert np.array_equal(r, cl.orc.process_query(dbn, p.dimensions, cl.elts, raw, q))
        assert oc.integer_decode(cl.decrypt(r[0]), cl.orc.t) == exp


def test_process_request_pinned_host_buffers_zero_copy(srv10):
    """Page-locked host buffers are read and written in place by the kernels (no staging copies); the replies must be
    the ones the staged path produces, call after call (the second and later calls replay a captured graph)."""
    import torch
    p, cl, vals, db, server = srv10
    gk, raw = _gk(cl)
    q_pin = torch.empty((1, 2, cl.orc.k, N), dtype=torch.int64).pin_memory()
    out_pin = torch.empty((1, server.ctx.reply_cts, 2, cl.orc.k, N), dtype=torch.int64).pin_memory()
    q_np, out_np = q_pin.numpy().view(np.uint64), out_pin.numpy().view(np.uint64)
    dbn = db.read_ntt(0, 10)
    for idx in (3, 7, 3, 9):
        pt = np.zeros(N, dtype=np.uint64); pt[idx] = 1
        q = cl.encrypt(pt)[None]
        q_np[...] = q
        out_np[...] = 0
        server.ProcessRequest(pb.Request([q_np], gk), out=out_np)
        want = cl.orc.process_query(dbn, p.dimensions, cl.elts, raw, q)
        assert np.array_equal(out_np[0], want), idx
        staged = server.ProcessRequest(pb.Request([q.copy()], gk)).reply[0]
        assert np.array_equal(staged, want), idx


def test_process_request_2dim():
    # server_test.cpp:209-260
    p = _params(82, 7680, 2)
    cl = _harness(p, seed=89)
    rng = np.random.default_rng(42)
    vals = [int(v) for v in rng.integers(0, 1 << 48, 82, dtype=np.int64)]
    db = pb.PIRDatabase.Create(vals, p)
    server = pb.PIRServer.Create(db, p)
    gk, raw = _gk(cl)
    assert p.dimensions == [10, 9] and db.calculate_indices(42) == [4, 6]
    m_inv = pow(pb.next_power_two(19), -1, cl.orc.t)
    pt = np.zeros(N, dtype=np.uint64); pt[4] = m_inv; pt[16] = m_inv
    q = cl.encrypt(pt)[None]
    resp = server.ProcessRequest(pb.Request([q], gk))
    assert resp.reply[0].shape[0] == cl.orc.ER * 2
    assert np.array_equal(resp.reply[0], cl.orc.process_query(db.read_ntt(0, 82), p.dimensions, cl.elts, raw, q))
    assert oc.integer_decode(cl.process_reply(resp.reply[0]), cl.orc.t) == vals[42]


def test_server_create_size_mismatch():
    p = _params(10, 0, 1)
    db = pb.PIRDatabase.Create(p)  # empty
    with pytest.raises(pb.PIRStatusError) as e:  # server.cpp:37-39
        pb.PIRServer.Create(db, p)
    assert e.value.code == pb.INVALID_ARGUMENT


@pytest.mark.parametrize("n,bits,elem,bpc,dbsize,d,indices",
                         [(4096, 24, 0, 0, 10, 1, [0]), (4096, 24, 0, 10, 9, 2, [1, 5]),
                          (4096, 24, 0, 6, 500, 2, [9, 125]), (4096, 24, 64, 10, 1200, 1, [0, 80, 81, 123, 777, 1199]),
                          (4096, 24, 289, 10, 1200, 1, [0, 47, 777, 1199]), (8192, 20, 1024, 0, 300, 2, [0, 299])])
def test_end_to_end_correctness(n, bits, elem, bpc, dbsize, d, indices):
    # correctness_test.cpp:82-113 (decomposition arm) + one N=8192 shape: client -> ProcessRequest -> client
    p = _params(dbsize, elem, d, n, bits, bpc)
    cl = _harness(p, seed=5)
    items = _random_items(p)
    db = pb.PIRDatabase.Create(items, p)
    server = pb.PIRServer.Create(db, p)
    gk, raw = _gk(cl)
    queries = [cl.create_query(i) for i in indices]
    resp = server.ProcessRequest(pb.Request(queries, gk))
    assert cl.process_response_strings(indices, resp.reply) == [items[i] for i in indices]
    dbn = db.read_ntt(0, p.num_pt)
    want0 = cl.orc.process_query(dbn, p.dimensions, cl.elts, raw, queries[0])
    assert np.array_equal(resp.reply[0], want0)


# ------------------------------------------------------------------------------------------------ sharding on one GPU
# (9000, 1, 4): a one-dimensional database over three query ciphertexts; shards expand only the trees that cover their
# plaintexts (shard 2 starts inside the second tree, shard 3 spans the second and third)
@pytest.mark.parametrize("dbsize,d,shards", [(82, 2, 2), (82, 2, 3), (200, 1, 4), (50, 3, 2), (9, 2, 4), (9000, 1, 4)])
def test_row_sharded_partials_reduce_to_unsharded_answer(dbsize, d, shards):
    import torch
    from pir_b200 import sharded
    p = _params(dbsize, 0, d, 4096, 20)
    cl = _harness(p, seed=21)
    items = _random_items(p)
    db = pb.PIRDatabase.Create(items, p)
    server = pb.PIRServer.Create(db, p)
    gk, raw = _gk(cl)
    q = cl.create_query(dbsize // 2)
    want = server.ProcessRequest(pb.Request([q], gk)).reply[0]
    coeffs = oc.encode_string_db(cl.params, items)
    partials = []
    for s in range(shards):
        sh = sharded.ShardServer(p, device=0, shard_index=s, shard_count=shards)
        sh.load_coeff(coeffs)
        sh.set_keys(gk)
        partials.append(sh.answer_partial(torch.from_numpy(q.view(np.int64)).cuda()[None]))
    stacked = torch.stack(partials)
    out = sh.reduce_finish(stacked, n_queries=1)
    got = out.cpu().numpy().view(np.uint64).reshape(want.shape)
    assert np.array_equal(got, want)
    assert ob.string_decode(cl.process_reply(got), cl.orc.ptb, p.bytes_per_item) == items[dbsize // 2]


# ------------------------------------------------------------------------------------------------ full-size properties
def test_scan_selects_database_rows_at_baseline_size():
    """BASELINE config 2 shape (2^16 x 288 B, d=2, t 24 bit: 1639 plaintexts, dims [41,40]); size-independent
    property: a selection vector whose NTT form is (1,0) at column j and 0 elsewhere makes the scan return
    row r = DB[r*40 + j] exactly (c0) and 0 (c1)."""
    import torch
    from pir_b200 import sharded
    ep = pb.GenerateEncryptionParams(4096, 24)
    p = pb.CreatePIRParameters(1 << 16, 288, 2, ep)
    assert (p.num_pt, p.dimensions) == (1639, [41, 40])
    sh = sharded.ShardServer(p, device=0)
    sh.db.fill_random(7)
    k = 2
    j = 13
    sv = torch.zeros((40, 2, k, N), dtype=torch.int64, device="cuda")
    sv[j, 0] = 1  # NTT of the constant polynomial 1 is all-ones
    rows = sh.scan(sv[None])  # [1][41][2][k][N] NTT form
    rows = rows.cpu().numpy().view(np.uint64)[0]
    for r in (0, 1, 20, 40):
        idx = r * 40 + j
        if idx < p.num_pt:
            assert np.array_equal(rows[r, 0], sh.db.read_ntt(idx, 1)[0]), r
        else:
            assert not rows[r, 0].any()
        assert not rows[r, 1].any()
    # linearity: scan(a + b) == scan(a) + scan(b) mod q
    rng = np.random.default_rng(0)
    q = np.array(ep.coeff_modulus[:k], dtype=np.uint64)
    a = np.stack([rng.integers(0, int(q[jj]), (40, 2, N), dtype=np.uint64) for jj in range(k)], axis=2)
    b = np.stack([rng.integers(0, int(q[jj]), (40, 2, N), dtype=np.uint64) for jj in range(k)], axis=2)
    s = (a + b) % q[None, None, :, None]
    f = lambda x: sh.scan(torch.from_numpy(np.ascontiguousarray(x).view(np.int64)).cuda()[None]).cpu().numpy().view(np.uint64)[0]
    ra, rb, rs = f(a), f(b), f(s)
    assert np.array_equal((ra + rb) % q[None, None, :, None], rs)


@pytest.mark.parametrize("n,bits,dbsize,d,nq", [(4096, 20, 82, 2, 4), (4096, 20, 82, 2, 7), (4096, 20, 300, 2, 5),
                                                (4096, 20, 37, 1, 6), (8192, 20, 50, 2, 4), (4096, 24, 1639, 2, 9)])
def test_batched_scan_matches_single_query_scan_and_oracle(n, bits, dbsize, d, nq):
    """Batches of >= 4 queries share one pass over the database (k_scan_batch2): every query's rows must equal what
    the single-query kernel returns for it, and the oracle's selection-vector x database row (database.cpp:185-194).
    Shapes cover a short last row, d=1 (one row), odd batch sizes (a half-empty query tile) and N=8192."""
    import torch
    from pir_b200 import sharded
    ep = pb.GenerateEncryptionParams(n, bits)
    p = pb.CreatePIRParameters(dbsize, 0, d, ep)
    sh = sharded.ShardServer(p, device=0)
    sh.db.fill_random(11)
    k = len(ep.coeff_modulus) - 1
    dimL = p.dimensions[-1]
    rng = np.random.default_rng(3)
    q = [int(x) for x in ep.coeff_modulus[:k]]
    sv = np.stack([rng.integers(0, q[j], (nq, dimL, 2, n), dtype=np.uint64) for j in range(k)], axis=3)
    d_sv = torch.from_numpy(np.ascontiguousarray(sv).view(np.int64)).cuda()
    batch = sh.scan(d_sv).cpu().numpy().view(np.uint64)
    for i in range(nq):
        single = sh.scan(d_sv[i:i + 1]).cpu().numpy().view(np.uint64)[0]
        assert np.array_equal(batch[i], single), i
    orc = ob.Oracle(n, list(ep.coeff_modulus), ep.plain_modulus)
    n_rows = batch.shape[1]
    for i, r in [(0, 0), (nq - 1, n_rows - 1), (nq // 2, n_rows // 2)]:
        first = r * dimL
        cnt = min(dimL, p.num_pt - first)
        want = orc.scan_row(sh.db.read_ntt(first, cnt), sv[i, :cnt])
        assert np.array_equal(batch[i, r], want), (i, r)


# ------------------------------------------------------------------------------------------------ golden fixtures
def _load_digest_module():
    import importlib.util
    here = os.path.dirname(os.path.abspath(__file__))
    spec = importlib.util.spec_from_file_location("make_oracle_digests",
                                                  os.path.join(here, "golden", "make_oracle_digests.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    with open(os.path.join(here, "golden", "oracle_digests.json")) as f:
        return mod, json.load(f)


class _CudaBackend:
    """substitute / shift / expand / answer through the product API, for tests/golden/make_oracle_digests.run_case"""

    def __init__(self, hp, db_limbs, elts, keys_flat):
        ep = pb.EncryptionParameters(hp.poly_modulus_degree, hp.plain_modulus, list(hp.coeff_modulus))
        self.p = pb.PIRParameters(num_items=hp.num_items, num_pt=hp.num_pt, dimensions=list(hp.dimensions),
                                  encryption_parameters=ep, bytes_per_item=hp.bytes_per_item,
                                  items_per_plaintext=hp.items_per_plaintext, bits_per_coeff=hp.bits_per_coeff)
        self.db = pb.PIRDatabase.Create(self.p)
        self.db.load_ntt(db_limbs)
        self.server = pb.PIRServer.Create(self.db, self.p)
        self.gk = pb.GaloisKeys(elts, keys_flat)
        self.db_limbs, self.ct_server = db_limbs, None

    def answer_ct(self, query, relin):
        if self.ct_server is None:  # the same database behind a context of the ciphertext-multiplication mode
            import dataclasses
            pc = dataclasses.replace(self.p, use_ciphertext_multiplication=True)
            dbc = pb.PIRDatabase.Create(pc)
            dbc.load_ntt(self.db_limbs)
            self.ct_server = pb.PIRServer.Create(dbc, pc)
        return self.ct_server.ProcessRequest(pb.Request([query], self.gk, relin_keys=relin)).reply[0][0]

    def substitute(self, ct, power):
        got = ct.copy()
        self.server.substitute_power_x_inplace(got, power, self.gk)
        return got

    def shift(self, ct, k):
        return self.server.multiply_inverse_power_of_x(ct, k)

    def expand(self, cts, total):
        return self.server.oblivious_expansion(cts, total, self.gk)

    def answer(self, query):
        return self.server.ProcessRequest(pb.Request([query], self.gk)).reply[0]


def test_cuda_path_reproduces_the_committed_golden_digests():
    """tests/golden/oracle_digests.json freezes the oracle's substitution / shift / expansion / reply for SHAKE-derived
    inputs; the CUDA path must produce byte-identical objects (same SHA-256) for N=4096 d=1/d=2, t 24-bit and N=8192 —
    including the replies of the ciphertext-multiplication mode with and without a relinearization key."""
    mod, want = _load_digest_module()
    for name, *args in mod.CASES:
        got = mod.run_case(name, *args, make_backend=_CudaBackend)
        assert got == want[name], name


def test_repeated_requests_replay_the_captured_graph(srv10):
    """The first ProcessRequest of a shape runs eagerly, the second captures a CUDA graph, later ones replay it:
    every reply must still match the oracle, also after the client (key handle) changes."""
    p, cl, vals, db, server = srv10
    gk, raw = _gk(cl)
    dbn = db.read_ntt(0, 10)
    for rep in range(5):
        pt = np.zeros(N, dtype=np.uint64); pt[rep] = 1
        q = cl.encrypt(pt)[None]
        r = server.ProcessRequest(pb.Request([q], gk)).reply[0]
        assert np.array_equal(r, cl.orc.process_query(dbn, p.dimensions, cl.elts, raw, q)), rep
    cl2 = _harness(p, seed=4242)
    gk2, raw2 = _gk(cl2)
    for rep in range(3):
        pt = np.zeros(N, dtype=np.uint64); pt[9 - rep] = 1
        q = cl2.encrypt(pt)[None]
        r = server.ProcessRequest(pb.Request([q], gk2)).reply[0]
        assert np.array_equal(r, cl2.orc.process_query(dbn, p.dimensions, cl2.elts, raw2, q)), rep
        assert oc.integer_decode(cl2.decrypt(r[0]), cl2.orc.t) == vals[9 - rep] * 16


def test_cpp_shim_end_to_end():
    """pir::PIRServer / pir::PIRDatabase C++ shim (pir_b200/cpp/pir_b200.hpp) over the C ABI: build/shim_test runs the
    reference-style client -> ProcessRequest -> client round trip and compares reply limbs with the oracle."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "build", "shim_test")
    if not os.path.exists(exe):
        subprocess.check_call(["make", "-C", root, "build/shim_test"])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "SHIM_TEST_OK" in out.stdout, out.stdout[-1500:] + out.stderr[-1500:]


# ------------------------------------------------------------------------------------------------ other engines / sizes
def _find_ntt_primes(bits, n, count):
    out, v = [], (1 << bits) - 2 * n + 1
    while len(out) < count:
        if ob.is_prime(v):
            out.append(v)
        v -= 2 * n
    return out


@pytest.mark.parametrize("n,bits,label", [(4096, 60, "60-bit moduli: corrected integer butterflies + 128-bit MACs"),
                                           (4096, 50, "50-bit moduli: corrected integer butterflies + 128-bit MACs"),
                                           (4096, 47, "47-bit moduli: lazy integer butterflies + 24-bit-split MACs"),
                                           (2048, 40, "N=2048 with two data moduli: FP64 engine at another size"),
                                           (16384, 44, "N=16384, k=3: FP64 engine, 128 KiB transforms")])
def test_custom_moduli_exercise_every_engine(n, bits, label):
    """Parity does not depend on the arithmetic engine: custom coefficient moduli force the integer fallbacks
    (moduli above 44 bits) and other transform sizes; expansion + multiply must still match the oracle limb for limb.
    (Noise is irrelevant here: inputs are random ring elements.)"""
    k = 2 if n != 16384 else 3
    mods = _find_ntt_primes(bits, n, k + 1)
    ep = pb.EncryptionParameters(n, ob.plain_modulus_batching(n, 20), mods)
    p = pb.CreatePIRParameters(23, 0, 2, ep)
    orc = ob.Oracle(n, mods, ep.plain_modulus)
    rng = np.random.default_rng(bits)
    coeffs = rng.integers(0, ep.plain_modulus, (p.num_pt, n), dtype=np.uint64)
    db = pb.PIRDatabase.Create(p)
    db.load_coeff(coeffs)
    want_db = np.stack([orc.plain_to_ntt(c) for c in coeffs])
    assert np.array_equal(db.read_ntt(0, p.num_pt), want_db), label
    server = pb.PIRServer.Create(db, p)
    elts = pb.generate_galois_elts(n)
    n_lvl = pb.ceil_log2(sum(p.dimensions))
    elts = elts[:n_lvl]
    keys = np.ascontiguousarray(np.stack([np.stack([np.stack([np.stack(
        [rng.integers(0, mods[i], n, dtype=np.uint64) for i in range(k + 1)]) for _ in range(2)]) for _ in range(k)])
        for _ in elts]))
    gk = pb.GaloisKeys(elts, keys.reshape(-1))
    q = np.stack([rng.integers(0, mods[j], n, dtype=np.uint64) for _ in range(2) for j in range(k)]).reshape(1, 2, k, n)
    got = server.ProcessRequest(pb.Request([q], gk)).reply[0]
    want = orc.process_query(want_db, p.dimensions, elts, keys.reshape(-1), q)
    assert got.shape == want.shape and np.array_equal(got, want), label


@pytest.mark.parametrize("n,bits", [(4096, 60), (4096, 47), (16384, 44)])
def test_ct_multiply_mode_with_custom_moduli(n, bits):
    """The ciphertext-multiplication mode next to the other arithmetic engines (integer NTTs for the data moduli too,
    N = 16384 with three data moduli): expansion + multiply + relinearization on random ring elements, limb for limb."""
    k = 2 if n != 16384 else 3
    mods = _find_ntt_primes(bits, n, k + 1)
    ep = pb.EncryptionParameters(n, ob.plain_modulus_batching(n, 20), mods)
    p = pb.CreatePIRParameters(11, 0, 2, ep, True)
    orc = ob.Oracle(n, mods, ep.plain_modulus)
    rng = np.random.default_rng(bits + 1)
    coeffs = rng.integers(0, ep.plain_modulus, (p.num_pt, n), dtype=np.uint64)
    db = pb.PIRDatabase.Create(p)
    db.load_coeff(coeffs)
    want_db = np.stack([orc.plain_to_ntt(c) for c in coeffs])
    server = pb.PIRServer.Create(db, p)
    elts = pb.generate_galois_elts(n)[:pb.ceil_log2(sum(p.dimensions))]

    def key_limbs(count):
        return np.ascontiguousarray(np.stack([np.stack([np.stack([np.stack(
            [rng.integers(0, mods[i], n, dtype=np.uint64) for i in range(k + 1)]) for _ in range(2)]) for _ in range(k)])
            for _ in range(count)]))
    keys, relin = key_limbs(len(elts)), key_limbs(1).reshape(-1)
    gk = pb.GaloisKeys(elts, keys.reshape(-1))
    qs = [np.stack([rng.integers(0, mods[j], n, dtype=np.uint64) for _ in range(2) for j in range(k)]).reshape(1, 2, k, n)
          for _ in range(2)]
    for rk in (relin, None):
        resp = server.ProcessRequest(pb.Request(qs, gk, relin_keys=rk))
        for q, r in zip(qs, resp.reply):
            want = orc.process_query_ct(want_db, p.dimensions, elts, keys.reshape(-1), q, rk)
            assert r.shape[1:] == want.shape and np.array_equal(r[0], want), (n, bits, rk is None)


def test_multiply_with_unused_selection_entries_and_empty_database():
    """database.cpp:183: the scan stops when the database runs out.  dims given by the caller need not be tight:
    [4,4] over 5 plaintexts leaves rows 2,3 empty and row 1 short; only the touched selection entries become NTT form."""
    ep = pb.GenerateEncryptionParams(4096, 20)
    p = pb.PIRParameters(num_items=5, num_pt=5, dimensions=[4, 4], encryption_parameters=ep, bytes_per_item=9728,
                         items_per_plaintext=1)
    orc = ob.Oracle(4096, ep.coeff_modulus, ep.plain_modulus)
    rng = np.random.default_rng(77)
    coeffs = rng.integers(0, ep.plain_modulus, (5, 4096), dtype=np.uint64)
    db = pb.PIRDatabase.Create(p)
    db.load_coeff(coeffs)
    sv = np.stack([np.stack([rng.integers(0, ep.coeff_modulus[j], 4096, dtype=np.uint64) for _ in range(2)
                             for j in range(2)]).reshape(2, 2, 4096) for _ in range(8)])
    want, sv_after = orc.db_multiply(np.stack([orc.plain_to_ntt(c) for c in coeffs]), [4, 4], sv)
    got_sv = sv.copy()
    got = db.multiply(got_sv)
    assert np.array_equal(got, want)
    assert np.array_equal(got_sv, sv_after)      # entries 2,3 of the first dimension stay in coefficient form
    empty = pb.PIRDatabase.Create(p)
    assert empty.multiply(sv.copy()).shape[0] == 0   # reference returns an empty vector (database.cpp:181-183)


def test_device_populate_and_shard_file_roundtrip(tmp_path):
    """pirb_db_load_items packs raw item bytes on the device exactly like StringEncoder (string_encoder.cpp:58-122),
    for several (bytes_per_item, bits_per_coeff) shapes incl. a short last plaintext; save()/load() round-trips."""
    for n, bits, elem, bpc, dbsize in [(4096, 20, 64, 0, 1200), (4096, 24, 289, 10, 777), (4096, 16, 1, 0, 5000),
                                       (8192, 20, 1024, 13, 100), (4096, 20, 9728, 0, 3)]:
        p = _params(dbsize, elem, 1, n, bits, bpc)
        cl = _harness(p)
        items = _random_items(p, seed=elem)
        db = pb.PIRDatabase.Create(items, p)            # device packing path (fixed-size items)
        assert db.size() == p.num_pt
        want = oc.db_to_ntt(cl.orc, oc.encode_string_db(cl.params, items))
        got = db.read_ntt(0, p.num_pt)
        assert np.array_equal(got, want), (n, bits, elem, bpc, dbsize)
    path = str(tmp_path / "shard.bin")
    db.save(path)
    db2 = pb.PIRDatabase.Create(p)
    db2.load(path)
    assert db2.size() == p.num_pt and np.array_equal(db2.read_ntt(0, p.num_pt), got)


# ------------------------------------------------------------------------------------------------ NVLink exchange flow
_PEER_FLOW = [(82, 2, 2, 1, 0), (82, 3, 3, 2, 0), (300, 4, 4, 0, 0), (3, 4, 1, 0, 0), (300, 2, 5, 2, 0), (300, 2, 5, 2, 1),
              (82, 3, 3, 2, 1), (300, 4, 2, 0, 1)]
# tensor-core exchange geometries: 20 queries per scan (two query tiles); a last dimension of 400 (four K chunks, one
# B buffer); empty shards; a last dimension of 1100, whose B operand fits only with 8-query tiles
_PEER_FLOW_TC = [(300, 4, 5, 5, 1, None), (1350, 2, 5, 5, 1, [4, 400]), (3, 4, 1, 0, 1, None),
                 (2150, 2, 5, 5, 1, [2, 1100])]


@pytest.mark.parametrize("dbsize,world,ql,sub,packed,dims",
                         [pytest.param(*r, None, id="-".join(map(str, r))) for r in _PEER_FLOW] +
                         [pytest.param(*r, id="-".join(map(str, r[:5])) + ("" if r[5] is None else "-dims%dx%d" % tuple(r[5])))
                          for r in _PEER_FLOW_TC])
def test_peer_memory_exchange_flow_matches_oracle(dbsize, world, ql, sub, packed, dims, monkeypatch):
    """pirb_dist_*: the row-sharded flow whose exchange is done by the kernels over peer memory (selection-vector NTT
    storing into every rank's slot, per-sub-batch flags, partial replies added by peer loads).  All ranks live in this
    process and on this one GPU (ShardGroup), which exercises exactly the kernels, flags and slot arithmetic of the
    one-process-per-GPU deployment.  Every rank's replies must equal the oracle's ProcessRequest on the unsharded
    database, limb for limb; two steps, so both exchange slots and the flag sequence numbers are used.  Shapes cover
    a short last row, ranks with fewer rows than others, empty shards (4 ranks over 2 rows), ragged sub-batches and more
    ranks than sub-batches.  (At most 4 ranks share the GPU here: every rank brings 3 library streams, and streams
    beyond CUDA_DEVICE_MAX_CONNECTIONS = 8 hardware queues per device can be serialised behind a spinning wait
    kernel — one rank per GPU, the deployment, is far below that.)"""
    import torch
    from pir_b200 import sharded
    if packed:
        # packed = 1: the last-dimension entries travel repacked into the tensor-core operand layout and every scan runs on the
        # tensor cores (normally chosen for shards of >= 1024 plaintexts; forced here on the small test database)
        monkeypatch.setenv("PIRB_TC_MIN_PT", "0")
    else:
        monkeypatch.setenv("PIRB_DIST_TC", "0")
    n = 4096
    ep = pb.GenerateEncryptionParams(n, 20)
    p = pb.CreatePIRParameters(dbsize, 0, 2, ep)
    if dims is not None:  # explicit dimensions: a long last dimension over a small database
        p = dataclasses.replace(p, dimensions=list(dims))
    mods = list(ep.coeff_modulus)
    k = len(mods) - 1
    rng = np.random.default_rng(dbsize * 31 + world)
    grp = sharded.ShardGroup(p, [0] * world, ql, sub)
    coeffs = rng.integers(0, ep.plain_modulus, (p.num_pt, n), dtype=np.uint64)
    grp.load_coeff(coeffs)
    orc = ob.Oracle(n, mods, ep.plain_modulus)
    db_ntt = np.stack([orc.plain_to_ntt(c) for c in coeffs])
    elts = [(n >> i) + 1 for i in range(12)]
    keys = np.stack([rng.integers(0, q, (len(elts), k, 2, n), dtype=np.uint64) for q in mods], axis=3)
    grp.set_keys(pb.GaloisKeys(elts, keys.reshape(-1)))
    n_ct = sum(p.dimensions) // n + 1
    for step in range(2):
        queries = np.stack([rng.integers(0, q, (world, ql, n_ct, 2, n), dtype=np.uint64) for q in mods[:k]], axis=4)
        outs = grp.answer([sharded.to_device(queries[r], "cuda:0") for r in range(world)])
        for r in range(world):
            got = sharded.to_host(outs[r])
            for i in range(ql):
                want = orc.process_query(db_ntt, p.dimensions, elts, keys.reshape(-1), queries[r, i])
                assert np.array_equal(got[i], want), (step, r, i)


# ------------------------------------------------------------------------------------------------ engines, wide moduli
@pytest.mark.parametrize("env", [{"PIRB_NTT_ENGINE": "0"}, {"PIRB_NTT_ENGINE": "1"}, {"PIRB_MAC_MODE": "0"},
                                 {"PIRB_MAC_MODE": "1"}, {"PIRB_KS_CLUSTER": "0"}, {"PIRB_TC_MIN": "0"},
                                 {"PIRB_TC_MIN_PT": "0"}, {"PIRB_GRAPHS": "0"},
                                 {"PIRB_NTT_ENGINE": "0", "PIRB_MAC_MODE": "0", "PIRB_KS_CLUSTER": "0"}])
def test_every_engine_variant_is_bit_identical(env, monkeypatch):
    """The library picks the fastest exact arithmetic the moduli allow (FP64 / lazy integer / corrected integer NTT
    engines, FP64 / 24-bit / 128-bit multiply-accumulate chains, cluster or three-launch key switch, tensor-core or
    CUDA-core batched scan, graph replay or eager launches).  All of them are exact, so forcing any of them must give the
    oracle's answer limb for limb: a batch of 5 queries on the reference's 2-dimensional test shape."""
    for kk, v in env.items():
        monkeypatch.setenv(kk, v)
    n = 4096
    ep = pb.GenerateEncryptionParams(n, 20)
    p = pb.CreatePIRParameters(82, 0, 2, ep)
    mods = list(ep.coeff_modulus)
    k = len(mods) - 1
    rng = np.random.default_rng(17)
    coeffs = rng.integers(0, ep.plain_modulus, (p.num_pt, n), dtype=np.uint64)
    db = pb.PIRDatabase(p)
    db.load_coeff(coeffs)
    server = pb.PIRServer.Create(db, p)
    orc = ob.Oracle(n, mods, ep.plain_modulus)
    db_ntt = np.stack([orc.plain_to_ntt(c) for c in coeffs])
    elts = [(n >> i) + 1 for i in range(12)]
    keys = np.stack([rng.integers(0, q, (len(elts), k, 2, n), dtype=np.uint64) for q in mods], axis=3)
    gk = pb.GaloisKeys(elts, keys.reshape(-1))
    queries = np.stack([rng.integers(0, q, (5, 1, 2, n), dtype=np.uint64) for q in mods[:k]], axis=3)
    for rep in range(2):  # second call replays the captured graph where graphs are on
        got = server.ProcessRequest(pb.Request([q for q in queries], gk)).reply
        for i in range(5):
            want = orc.process_query(db_ntt, p.dimensions, elts, keys.reshape(-1), queries[i])
            assert np.array_equal(got[i], want), (env, rep, i)


@pytest.mark.parametrize("dims", [[600], [300, 2]])
def test_sixty_bit_moduli_keep_lazy_accumulation_chains_exact(dims):
    """Moduli up to 2^61 are accepted (SEAL allows user moduli up to 60 bits); products are then below 2^120 and a
    128-bit lazy accumulator wraps after 256 terms.  A dimension of 600 (scan) or 300 (upper dimension) must therefore
    be split into exact chains: pirb_db_multiply against the oracle, N=2048, one 60-bit data modulus."""
    n = 2048
    mods = [0xfffffffffffc001, 0xffffffffffe8001]       # data modulus, special prime: 60-bit, = 1 mod 2N
    t = int(pb.GenerateEncryptionParams(4096, 20).plain_modulus)
    assert all((q - 1) % (2 * n) == 0 for q in mods)
    num_pt = 600
    ep = pb.EncryptionParameters(n, t, mods)
    p = pb.PIRParameters(num_items=num_pt, num_pt=num_pt, dimensions=list(dims), bytes_per_item=0, items_per_plaintext=1,
                         bits_per_coeff=0, encryption_parameters=ep)
    rng = np.random.default_rng(23)
    orc = ob.Oracle(n, mods, t)
    db_ntt = rng.integers(0, mods[0], (num_pt, 1, n), dtype=np.uint64)
    db = pb.PIRDatabase(p)
    db.load_ntt(db_ntt)
    sv = rng.integers(0, mods[0], (sum(dims), 2, 1, n), dtype=np.uint64)
    want, sv_after = orc.db_multiply(db_ntt, dims, sv)
    got_sv = sv.copy()
    got = db.multiply(got_sv)
    assert np.array_equal(got, want)
    assert np.array_equal(got_sv, sv_after)


# ------------------------------------------------------------------------------------------------ parity at full size
@pytest.mark.parametrize("workload,nq", [("cfg4", 1), ("cfg4", 8), ("cfg3", 1), ("cfg3", 4), ("cfg5b", 1)])
def test_full_size_databases_sampled_parity(workload, nq):
    """BASELINE configs[3] (2^22 x 256 B, 6.7 GiB), configs[2] (N=8192, 2^20 x 1 KiB, 13.5 GiB) and configs[4] d=2
    (2^24 x 256 B, 27 GiB) at their real sizes on one GPU, synthetic NTT-form database.  The oracle cannot process
    gigabytes in a test, so the chain is checked in pieces that together cover every kernel at full grid size
    (sharded.sampled_parity): the full expansion + selection-vector NTT of a query; the scan of the whole database with
    the first, a middle and the short last row recomputed by the oracle from the device's database; the upper dimension
    recomputed by the oracle from ALL device rows.  nq > 1 answers a batch (tensor-core scan) and checks query 0 and
    that every query of the batch equals its single-query answer."""
    import torch
    import bench
    from pir_b200 import sharded
    items, size, d, n, bits, _ = bench.WORKLOADS[workload]
    p = pb.CreatePIRParameters(items, size, d, pb.GenerateEncryptionParams(n, bits))
    ep = p.encryption_parameters
    mods = list(ep.coeff_modulus)
    free, _total = torch.cuda.mem_get_info()
    need = p.num_pt * (len(mods) - 1) * n * 8 * (1.8 if nq > 1 else 1.1) + (8 << 30)
    if free < need:
        pytest.skip("not enough free device memory for %s" % workload)
    srv = sharded.ShardServer(p, device=0)
    srv.db.fill_random(5)
    queries, elts, keys = bench.synth_inputs(n, mods, list(p.dimensions), nq, 31)
    srv.set_keys(pb.GaloisKeys(elts, keys.reshape(-1)))
    d_q = sharded.to_device(queries, "cuda:0")
    replies = sharded.to_host(srv.answer(d_q))
    orc = ob.Oracle(n, mods, ep.plain_modulus)
    ok, desc = sharded.sampled_parity(srv, orc, p, elts, keys, queries[0], replies[0])
    assert ok, desc
    for i in range(1, nq):
        single = sharded.to_host(srv.answer(d_q[i:i + 1]))[0]
        assert np.array_equal(replies[i], single), i


# ------------------------------------------------------------------------------------------------ ciphertext-multiplication mode
def _selection_vector(cl, dims, indices):
    cts = []
    for d, dim in enumerate(dims):
        for i in range(dim):
            pt = np.zeros(cl.orc.N, dtype=np.uint64)
            if i == indices[d]:
                pt[0] = 1
            cts.append(cl.encrypt(pt))
    return np.stack(cts)


@pytest.mark.parametrize("n,bits,dbsize,d,idx", [(4096, 16, 10, 1, 7), (4096, 16, 16, 2, 11), (4096, 16, 82, 2, 42),
                                                  (8192, 20, 27, 3, 2), (8192, 20, 117, 3, 17)])
def test_ct_multiply_mode_db_multiply_matches_oracle(n, bits, dbsize, d, idx):
    """database_test.cpp:343-388, CTMultiply arm (use_ciphertext_multiplication, relinearization keys given): the single
    result ciphertext bit-exact against the oracle's Evaluator::multiply + relinearize_inplace restatement, decrypting
    to the selected item; without keys (server.cpp:185-190) the result keeps one more polynomial per upper dimension."""
    p = _params(dbsize, 0, d, n, bits, ct_mult=True)
    cl = _harness(p, seed=11)
    items = _random_items(p)
    db = pb.PIRDatabase.Create(items, p)
    db_ntt = oc.db_to_ntt(cl.orc, oc.encode_string_db(cl.params, items))
    assert np.array_equal(db.read_ntt(0, p.num_pt), db_ntt)
    sv = _selection_vector(cl, p.dimensions, oc.calculate_indices(cl.params, idx))
    before = sv.copy()
    got = db.multiply(sv, cl.relin)
    assert np.array_equal(sv, before)  # database.cpp:188: left in coefficient form in this mode
    want = cl.orc.db_multiply_ct(db_ntt, p.dimensions, sv, cl.relin)
    assert got.shape == (1, 2, cl.orc.k, n) and np.array_equal(got[0], want)
    res = cl.process_reply_ct(got)
    assert ob.string_decode(res, cl.orc.ptb, p.bytes_per_item) == items[idx]
    # no relinearization keys: d + 1 polynomials (d = 1: the plain two)
    got_nr = db.multiply(sv)
    want_nr = cl.orc.db_multiply_ct(db_ntt, p.dimensions, sv, None)
    assert got_nr.shape == (1, 2 if d == 1 else d + 1, cl.orc.k, n) and np.array_equal(got_nr[0], want_nr)
    with pytest.raises(pb.PIRStatusError) as e:  # database.cpp:297-300
        db.multiply(np.ascontiguousarray(sv[:-1]), cl.relin)
    assert e.value.code == pb.INVALID_ARGUMENT


@pytest.mark.parametrize("n,bits,elem,bpc,dbsize,d,indices",
                         [(4096, 24, 0, 0, 10, 1, [0]), (4096, 16, 0, 10, 9, 2, [1, 5]),
                          (4096, 16, 0, 6, 500, 2, [9, 125]), (8192, 42, 0, 0, 87, 2, [5, 33, 86]),
                          (4096, 16, 64, 10, 1200, 1, [0, 80, 81, 123, 777, 1199]),
                          (4096, 16, 0, 6, 500, 2, [9, 125, 0, 250, 499])])
def test_ct_multiply_mode_end_to_end_matches_oracle(n, bits, elem, bpc, dbsize, d, indices, monkeypatch):
    """correctness_test.cpp:94-105 (use_ciphertext_multiplication == true): client -> PIRServer::ProcessRequest ->
    client, every reply bit-exact against the oracle, the whole batch of queries in one device call.  A batch of 4 or
    more queries at d >= 2 takes the tensor-core last-dimension scan, here even on a small database."""
    if d >= 2 and len(indices) >= 4:
        monkeypatch.setenv("PIRB_TC_MIN_PT", "0")
    p = _params(dbsize, elem, d, n, bits, bpc, ct_mult=True)
    cl = _harness(p, seed=5)
    items = _random_items(p)
    db = pb.PIRDatabase.Create(items, p)
    server = pb.PIRServer.Create(db, p)
    db_ntt = oc.db_to_ntt(cl.orc, oc.encode_string_db(cl.params, items))
    queries = [cl.create_query(i) for i in indices]
    gk, raw = _gk(cl)
    resp = server.ProcessRequest(pb.Request(query=queries, galois_keys=gk, relin_keys=cl.relin))
    assert len(resp.reply) == len(indices)
    for q, r in zip(queries, resp.reply):
        want = cl.orc.process_query_ct(db_ntt, p.dimensions, cl.elts, raw, q, cl.relin)
        assert r.shape == (1, 2, cl.orc.k, n) and np.array_equal(r[0], want)
    assert cl.process_response_strings(indices, resp.reply) == [items[i] for i in indices]
    if d == 2 and n == 4096:  # a request without relinearization keys: size-3 replies
        resp3 = server.ProcessRequest(pb.Request(query=queries[:1], galois_keys=gk))
        want3 = cl.orc.process_query_ct(db_ntt, p.dimensions, cl.elts, raw, queries[0], None)
        assert resp3.reply[0].shape == (1, 3, cl.orc.k, n) and np.array_equal(resp3.reply[0][0], want3)
        assert cl.process_response_strings(indices[:1], resp3.reply) == [items[indices[0]]]


def test_ct_multiply_mode_process_request_2dim_and_wire():
    """server_test.cpp:209-260 with GetParam() == true (reply is one ciphertext of size 2: "Were relin keys used?"),
    then the same request in its serialized form (relin_keys field used, server.cpp:53-58)."""
    from pir_b200 import wire
    p = _params(82, 7680, 2, ct_mult=True)
    cl = _harness(p, seed=89)
    rng = np.random.default_rng(42)
    vals = [int(v) for v in rng.integers(0, 1 << 48, 82, dtype=np.int64)]
    db = pb.PIRDatabase.Create(vals, p)
    server = pb.PIRServer.Create(db, p)
    m_inv = pow(ob.next_power_two(19), -1, p.encryption_parameters.plain_modulus)
    pt = np.zeros(N, dtype=np.uint64); pt[4] = m_inv; pt[16] = m_inv
    q = cl.encrypt(pt)[None]
    gk, raw = _gk(cl)
    resp = server.ProcessRequest(pb.Request(query=[q], galois_keys=gk, relin_keys=cl.relin))
    assert resp.reply[0].shape == (1, 2, cl.orc.k, N)
    assert oc.integer_decode(cl.process_reply_ct(resp.reply[0]), p.encryption_parameters.plain_modulus) == vals[42]
    relin_blob = wire.save_galois_keys(pb.GaloisKeys([1], cl.relin), p.encryption_parameters)  # slot 0 of a KSwitchKeys
    blob = wire.serialize_request([q], gk, p, relin_keys=relin_blob)
    back = wire.parse_response(server.ProcessRequestBytes(blob), p)
    assert np.array_equal(back.reply[0], resp.reply[0])
    # the entry points of the re-encoder path refuse a context of this mode
    import ctypes as C
    from pir_b200 import _lib
    out = np.zeros((1, 2, cl.orc.k, N), dtype=np.uint64)
    rc = _lib.lib().pirb_answer(server.ctx.h, server._keys(gk).h, C.c_void_p(q.ctypes.data), 1, 1,
                                C.c_void_p(out.ctypes.data))
    assert rc == pb.INVALID_ARGUMENT and "ciphertext-multiplication" in _lib.last_error()
