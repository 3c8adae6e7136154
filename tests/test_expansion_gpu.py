"""Oblivious expansion on every key-switch kernel the library can select, at every modulus width it supports.

Each tree level of the expansion is one key switch per node (Galois automorphism, key products, mod-down by the special
prime P) followed by the SealPIR butterfly.  Three implementations exist (pir_b200/csrc/kernels_cluster.cu,
kernels_ntt.cu, kernels_stream.cu) and the choice depends on the parameter set and on the level's width:

- `k_ks_level_cluster2<LN,K>` (second generation, cluster of k+1 CTAs): FP64 engine (every modulus <= 44 bits),
  N = 2048 / 4096, k <= 2, and a level of at least 2*SMs/(k+1) nodes;
- `k_ks_level_cluster<LN,ENG,MAC>` (first generation, cluster of 2(k+1) CTAs): the other levels, whenever the cluster
  has at most 16 CTAs and its shared memory fits;
- three launches (`k_ks_digits`, `k_ks_mac_intt`, `k_ks_combine`): everything else, and PIRB_KS_CLUSTER=0.

The engine (FP64 / lazy integer / corrected integer butterflies) and the multiply-accumulate (FP64 / 24-bit-split
Karatsuba / 128-bit) follow the widest modulus.  The rows below are parameter sets chosen so that together they launch
every instantiation; `_predicted_kernels` mirrors the dispatch and one test asserts, from a torch.profiler trace, that
each row launches exactly the kernels predicted.  Every other test compares with the CPU oracle, limb for limb: the
device-resident expansion + selection-vector NTT (`pirb_expand_ntt_dev`, eager, graph capture and graph replay), the
coefficient-form expansion (`pirb_expand`, single and vector overloads) and the substitution (`pirb_substitute`, one
node in substitution mode) for every Galois element.  Inputs are random ring elements (noise is irrelevant), uniform or
at the edges the FP64 bounds care about: limbs in the top 1/64 of [0, q), all q - 1, or sparse q - 1.
"""
import gc
import os
import re
import subprocess
import sys
import textwrap
import zlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import pir_b200 as pb
from oracle import binding as ob
from oracle import client as oc

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------------------ parameter sets
def _find_ntt_primes(bits, n, count):
    out, v = [], (1 << bits) - 2 * n + 1
    while len(out) < count:
        if ob.is_prime(v):
            out.append(v)
        v -= 2 * n
    return out


# id -> (N, moduli (data moduli, then the special prime), PIRB_KS_CLUSTER=0).  _find_ntt_primes returns descending
# primes, so the special prime is the smallest of its width.
ROWS = {
    "n4096": (4096, lambda: ob.bfv_default(4096), False),
    "q44-n4096": (4096, lambda: _find_ntt_primes(44, 4096, 3), False),
    # a data modulus above a key-level modulus (digits re-reduced mod m_I), and P much larger than q_1 in the mod-down
    "mix-n4096": (4096, lambda: _find_ntt_primes(44, 4096, 1) + _find_ntt_primes(32, 4096, 1)
                  + _find_ntt_primes(40, 4096, 1), False),
    "q44k1-n4096": (4096, lambda: _find_ntt_primes(44, 4096, 2), False),
    "q44k1-n2048": (2048, lambda: _find_ntt_primes(44, 2048, 2), False),
    "q44-n2048": (2048, lambda: _find_ntt_primes(44, 2048, 3), False),
    "q30k3-n4096": (4096, lambda: _find_ntt_primes(30, 4096, 4), False),
    "q30k4-n4096": (4096, lambda: _find_ntt_primes(30, 4096, 5), False),
    "q30k7-n4096": (4096, lambda: _find_ntt_primes(30, 4096, 8), False),
    "q30k8-n4096": (4096, lambda: _find_ntt_primes(30, 4096, 9), False),
    "n8192": (8192, lambda: ob.bfv_default(8192), False),
    "q44k3-n8192": (8192, lambda: _find_ntt_primes(44, 8192, 4), False),
    "q44k1-n8192": (8192, lambda: _find_ntt_primes(44, 8192, 2), False),
    "q44k5-n8192": (8192, lambda: _find_ntt_primes(44, 8192, 6), False),
    "q45-n4096": (4096, lambda: _find_ntt_primes(45, 4096, 3), False),
    "q49-n4096": (4096, lambda: _find_ntt_primes(49, 4096, 3), False),
    "q50-n4096": (4096, lambda: _find_ntt_primes(50, 4096, 3), False),
    "q48-n8192": (8192, lambda: _find_ntt_primes(48, 8192, 5), False),
    "q49-n8192": (8192, lambda: _find_ntt_primes(49, 8192, 5), False),
    "q60-n2048": (2048, lambda: _find_ntt_primes(60, 2048, 3), False),
    "n16384": (16384, lambda: ob.bfv_default(16384), False),
    "q44k3-n16384": (16384, lambda: _find_ntt_primes(44, 16384, 4), False),
    "q44-n4096-forced": (4096, lambda: _find_ntt_primes(44, 4096, 3), True),
    "q44k1-n2048-forced": (2048, lambda: _find_ntt_primes(44, 2048, 2), True),
}


def _row(row):
    n, mods, forced = ROWS[row]
    mods = [int(q) for q in mods()]
    return n, mods, forced


def _max_bits(mods):
    return max(q.bit_length() for q in mods)


def _is_big(n, mods):
    """Rows whose oracle key switch costs 5 ms or more: only narrow trees, plus the two-tree shape with one query."""
    return n >= 8192 or len(mods) - 1 >= 3


# ------------------------------------------------------------------------------------------------ the dispatch
ENG_INT, ENG_LAZY, ENG_FP64 = 0, 1, 2
MAC_WIDE, MAC_INT24, MAC_FP64 = 0, 1, 2
ENG_NAMES = {ENG_INT: "INT", ENG_LAZY: "LAZY", ENG_FP64: "FP64"}
MAC_NAMES = {MAC_WIDE: "WIDE", MAC_INT24: "INT24", MAC_FP64: "FP64"}


def _engine(n, mods):
    """context.cu: the NTT engine and the MAC from the widest modulus (special prime included)."""
    bits, logn = _max_bits(mods), n.bit_length() - 1
    eng = ENG_FP64 if bits <= 44 else (ENG_LAZY if bits <= 62 - logn - 1 else ENG_INT)
    mac = MAC_FP64 if bits <= 44 else (MAC_INT24 if bits <= 48 else MAC_WIDE)
    return eng, mac


def _cluster_smem(n, k, eng):
    """ks_cluster_smem: (k+1)/2 digit buffers, the accumulator, and for FP64 at N <= 4096 the staged twiddle table and
    its mbarrier."""
    tws = eng == ENG_FP64 and n <= 4096
    return ((k + 1) // 2 + 1 + (1 if tws else 0)) * n * 8 + (16 if tws else 0)


def _cluster_supported(n, k, eng):
    return 2 * (k + 1) <= 16 and _cluster_smem(n, k, eng) <= 227 * 1024 and 2048 <= n <= 16384


def _cluster2_supported(n, k, eng):
    return eng == ENG_FP64 and n in (2048, 4096) and k <= 2


def _level_nodes(n, dim_sum, nq):
    """Nodes of every tree level: queries x live trees x 2^j (get_plan: tree t expands min(N, dim_sum - t*N) items)."""
    items = [min(n, max(0, dim_sum - t * n)) for t in range(dim_sum // n + 1)]
    logm = [pb.ceil_log2(i) if i else 0 for i in items]
    return [nq * sum(1 for lm in logm if lm > j) << j for j in range(max(logm))]


def _predicted_kernels(n, mods, forced, nodes_per_level, sms):
    """The set of key-switch kernels run_expand / launch_ks_level_cluster launch for these levels."""
    k, logn = len(mods) - 1, n.bit_length() - 1
    eng, mac = _engine(n, mods)
    cluster = not forced and _cluster_supported(n, k, eng)
    out = set()
    for nodes in nodes_per_level:
        if not nodes:
            continue
        if not cluster:
            out |= {"k_ks_digits<%d,%d>" % (logn, eng), "k_ks_mac_intt<%d,%d>" % (logn, eng), "k_ks_combine"}
        elif _cluster2_supported(n, k, eng) and nodes >= 2 * sms // (k + 1):
            out.add("k_ks_level_cluster2<%d,%d>" % (logn, k))
        else:
            out.add("k_ks_level_cluster<%d,%d,%d>" % (logn, eng, mac))
    return out


def _describe(name, n, k):
    """Readable form of a kernel name for the coverage report."""
    m = re.match(r"(\w+)<([\d,]+)>", name)
    if not m:
        return name
    args = [int(a) for a in m.group(2).split(",")]
    if m.group(1) == "k_ks_level_cluster":
        return "k_ks_level_cluster<%d,%s,%s> (cluster of %d CTAs, %d KiB)" % (
            args[0], ENG_NAMES[args[1]], MAC_NAMES[args[2]], 2 * (k + 1), _cluster_smem(n, k, args[1]) // 1024)
    if m.group(1) == "k_ks_level_cluster2":
        return "k_ks_level_cluster2<%d,%d>" % tuple(args)
    return "%s<%d,%s>" % (m.group(1), args[0], ENG_NAMES[args[1]])


# ------------------------------------------------------------------------------------------------ inputs
def _limbs(fill, q, shape, rng):
    """Residues mod q: uniform; top (every limb in [q - q/64, q)); qminus1 (every limb q - 1); sparse (zeros with about
    one limb in 256 at q - 1)."""
    if fill == "uniform":
        return rng.integers(0, q, shape, dtype=np.uint64)
    if fill == "top":
        return rng.integers(q - q // 64, q, shape, dtype=np.uint64)
    if fill == "qminus1":
        return np.full(shape, q - 1, dtype=np.uint64)
    assert fill == "sparse"
    return np.where(rng.random(shape) < 1 / 256, np.uint64(q - 1), np.uint64(0))


def _key_fill(fill):
    """Keys at the top of their range for the edge fills, uniform otherwise."""
    return "top" if fill in ("top", "qminus1") else "uniform"


_KEYS = {}


def _keys(row, n, mods, fill):
    """Galois keys of every element, [elts][k][2][k+1][N] (limb i mod mods[i]); the last row's keys are cached."""
    key = (row, _key_fill(fill))
    if key not in _KEYS:
        _KEYS.clear()
        rng = np.random.default_rng(zlib.crc32(repr(key).encode()))
        elts = pb.generate_galois_elts(n)
        k = len(mods) - 1
        keys = np.stack([_limbs(_key_fill(fill), q, (len(elts), k, 2, n), rng) for q in mods], axis=3)
        _KEYS[key] = (elts, np.ascontiguousarray(keys).reshape(-1))
    return _KEYS[key]


def _queries(fill, mods, nq, n_ct, n, seed):
    """[nq][n_ct][2][k][N], limb j mod mods[j]."""
    rng = np.random.default_rng(seed)
    k = len(mods) - 1
    return np.ascontiguousarray(np.stack([_limbs(fill, mods[j], (nq, n_ct, 2, n), rng) for j in range(k)], axis=3))


def _params(n, mods, dim_sum):
    """dims [dim_sum] for dim_sum 1, else two dimensions summing to dim_sum; one plaintext (the expansion does not read
    the database)."""
    ep = pb.EncryptionParameters(n, ob.plain_modulus_batching(n, 20), mods)
    dims = [1] if dim_sum == 1 else [dim_sum // 2, dim_sum - dim_sum // 2]
    return pb.PIRParameters(num_items=1, num_pt=1, dimensions=dims, encryption_parameters=ep, bytes_per_item=0,
                            items_per_plaintext=1, bits_per_coeff=0)


def _shard(p, gk, monkeypatch, forced):
    from pir_b200 import sharded
    if forced:
        monkeypatch.setenv("PIRB_KS_CLUSTER", "0")  # read at context creation
    srv = sharded.ShardServer(p, device=0)
    if forced:
        monkeypatch.delenv("PIRB_KS_CLUSTER")
    srv.set_keys(gk)
    return srv


def _expand_ntt_into(srv, d_q, out):
    """ShardServer.expand_ntt into a caller-owned buffer: the same device pointers on every call, so that the second
    call captures the graph of pirb_expand_ntt_dev and the third replays it."""
    from pir_b200 import _lib
    from pir_b200.api import _check
    from pir_b200.sharded import _dp
    st = srv._enter()
    _check(_lib.lib().pirb_expand_ntt_dev(srv.ctx.h, srv.keys.h, _dp(d_q), d_q.shape[0], d_q.shape[1], _dp(out), st))
    srv._exit()


# ------------------------------------------------------------------------------------------------ the oracle
_POOL = ThreadPoolExecutor(max_workers=max(1, min(32, os.cpu_count() or 1)))  # the oracle's ctypes calls drop the GIL


def _oracle_check(n, mods, elts, keys, cts, total, single, got, ntt, tag):
    """Expand `cts` with the oracle (one Oracle per job) and compare with `got` ([total][2][k][N]); NTT form if ntt.
    Returns None or a description of the first difference."""
    orc = ob.Oracle(n, mods, ob.plain_modulus_batching(n, 20))
    want = orc.expand(cts, total, elts, keys, single=single)
    for i in range(total):
        w = orc.ct_to_ntt(want[i]) if ntt else want[i]
        if not np.array_equal(got[i], w):
            bad = np.argwhere(got[i] != w)
            return "%s: item %d differs at %d limbs, first (poly, modulus, coefficient) %s" % (
                tag, i, len(bad), tuple(int(x) for x in bad[0]))
    return None


def _run_jobs(jobs):
    errs = [e for e in _POOL.map(lambda a: _oracle_check(*a), jobs) if e]
    assert not errs, "\n".join(errs[:8])


# ------------------------------------------------------------------------------------------------ the matrix
TWO_TREE = "N+37"
FULL = "N"


def _shapes(n, mods):
    """(queries, dim_sum) per row.  Narrow rows: 300 items (9 levels of 1-256 nodes), 5 queries x 40 items (levels of
    5-160 nodes: one expansion crosses the generation threshold), 3 queries x N+37 (two trees, the second ragged),
    2 queries x N (the second ciphertext expands to nothing), 1 and 2 items (zero and one level).  Rows with an
    expensive oracle: 5 x 40, 1 x 64, 1 and 2 items, and one query x N+37 (not at N = 16384, whose 16384-item tree
    needs more workspace than a GPU has at k = 8 and repeats the three-launch path of the narrow shapes at k = 3)."""
    if not _is_big(n, mods):
        return [(1, 300), (5, 40), (3, TWO_TREE), (2, FULL), (1, 1), (1, 2)]
    out = [(5, 40), (1, 64), (1, 1), (1, 2)]
    if n < 16384:
        out.append((1, TWO_TREE))
    return out


def _dim_sum(n, spec):
    return n + 37 if spec == TWO_TREE else (n if spec == FULL else spec)


def _edge_row(row, n, mods):
    """FP64 rows at the 44-bit ceiling of the FP64 engine."""
    return _engine(n, mods)[0] == ENG_FP64 and _max_bits(mods) == 44


def _cases():
    out = []
    for row in ROWS:
        n, mods, forced = _row(row)
        shapes = _shapes(n, mods)
        for nq, spec in shapes:
            out.append((row, nq, spec, "uniform"))
        out.append((row, 5, 40, "sparse"))
        if _edge_row(row, n, mods):
            wide = [(nq, s) for nq, s in shapes if s in (300, 64, 40)]
            for fill in ("top", "qminus1"):
                out += [(row, nq, s, fill) for nq, s in (wide[:1] if forced else wide)]
    return out


CASES = _cases()


def _case_id(c):
    row, nq, spec, fill = c
    return "%s-q%d-s%s-%s" % (row, nq, spec, fill)


@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_expand_ntt_matches_oracle(case, monkeypatch):
    """ShardServer.expand_ntt (pirb_expand_ntt_dev: expansion + selection-vector NTT) three times on the same device
    buffers with new content each time — eager, graph capture, graph replay — every query and every item against the
    oracle's expansion followed by ct_to_ntt.  The one-query two-tree shape of the expensive rows checks the ragged tree
    against the oracle's single-ciphertext expansion of the second ciphertext (trees are independent) and the full
    tree against a PIRB_KS_CLUSTER=0 context of the same row."""
    import torch
    row, nq, spec, fill = case
    n, mods, forced = _row(row)
    k = len(mods) - 1
    dim_sum = _dim_sum(n, spec)
    p = _params(n, mods, dim_sum)
    elts, keys = _keys(row, n, mods, fill)
    gk = pb.GaloisKeys(elts, keys)
    srv = _shard(p, gk, monkeypatch, forced)
    split = _is_big(n, mods) and spec == TWO_TREE
    ref = _shard(p, gk, monkeypatch, True) if split else None
    n_ct = dim_sum // n + 1
    assert srv.ctx.query_cts == n_ct and srv.ctx.dim_sum == dim_sum
    d_q = torch.empty((nq, n_ct, 2, k, n), dtype=torch.int64, device="cuda")
    out = torch.empty((nq, dim_sum, 2, k, n), dtype=torch.int64, device="cuda")
    out_ref = torch.empty_like(out) if split else None
    for call in range(3):
        q = _queries(fill, mods, nq, n_ct, n, seed=1000 * call + nq + dim_sum)
        d_q.copy_(torch.from_numpy(q.view(np.int64)))
        out.fill_(-1)
        _expand_ntt_into(srv, d_q, out)
        if split:
            _expand_ntt_into(ref, d_q, out_ref)
        torch.cuda.synchronize()
        jobs = []
        for i in range(nq):
            tag = "call %d query %d" % (call, i)
            if split:
                assert torch.equal(out[i, :n], out_ref[i, :n]), tag + ": full tree differs from the three-launch path"
                got = out[i, n:].cpu().numpy().view(np.uint64)
                jobs.append((n, mods, elts, keys, q[i, 1], dim_sum - n, True, got, True, tag + " ragged tree"))
            else:
                got = out[i].cpu().numpy().view(np.uint64)
                jobs.append((n, mods, elts, keys, q[i], dim_sum, False, got, True, tag))
        _run_jobs(jobs)
    del out, out_ref, d_q, srv, ref
    gc.collect()
    torch.cuda.empty_cache()


def _coeff_cases():
    out = []
    for row in ROWS:
        n, mods, forced = _row(row)
        out.append((row, "uniform"))
        if _edge_row(row, n, mods) and not forced:
            out.append((row, "top"))
    return out


@pytest.mark.parametrize("row,fill", _coeff_cases(), ids=lambda v: v if isinstance(v, str) else None)
def test_coefficient_form_expansion_and_substitution_match_oracle(row, fill, monkeypatch):
    """PIRServer.oblivious_expansion (pirb_expand, coefficient form) on the one-query shapes — single-ciphertext and
    vector overloads — and substitute_power_x_inplace (one node in substitution mode) for every Galois element."""
    n, mods, forced = _row(row)
    k = len(mods) - 1
    elts, keys = _keys(row, n, mods, fill)
    gk = pb.GaloisKeys(elts, keys)
    orc = ob.Oracle(n, mods, ob.plain_modulus_batching(n, 20))
    jobs = []
    for nq, spec in _shapes(n, mods):
        if nq != 1 or spec in (TWO_TREE, FULL):
            continue
        total = _dim_sum(n, spec)
        p = _params(n, mods, total)
        if forced:
            monkeypatch.setenv("PIRB_KS_CLUSTER", "0")
        db = pb.PIRDatabase(p)
        monkeypatch.delenv("PIRB_KS_CLUSTER", raising=False)
        db.fill_random(total)
        server = pb.PIRServer.Create(db, p)
        q = _queries(fill, mods, 1, 1, n, seed=total)[0]
        got1 = server.oblivious_expansion(q[0], total, gk)
        jobs.append((n, mods, elts, keys, q[0], total, True, got1, False, "single, %d items" % total))
        gotv = server.oblivious_expansion(q, total, gk)
        jobs.append((n, mods, elts, keys, q, total, False, gotv, False, "vector, %d items" % total))
    _run_jobs(jobs)
    rng = np.random.default_rng(7)
    ct = np.ascontiguousarray(np.stack([_limbs(fill, mods[j], (2, n), rng) for j in range(k)], axis=1))
    for g in elts:
        got = ct.copy()
        server.substitute_power_x_inplace(got, g, gk)
        want = orc.substitute(ct, g, elts, keys)
        assert np.array_equal(got, want), "substitution by x -> x^%d" % g


# ------------------------------------------------------------------------------------------------ kernel coverage
def test_every_row_launches_the_predicted_key_switch_kernels(monkeypatch, capsys):
    """The first expand_ntt call of a fresh context per row (5 queries x 40 items: levels of 5 to 160 nodes), traced by
    torch.profiler: the set of k_ks_* kernels launched must equal the prediction of _predicted_kernels.  Prints every
    instantiation reached."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    reached = {}
    for row in ROWS:
        n, mods, forced = _row(row)
        k = len(mods) - 1
        nq, dim_sum = 5, 40
        elts, keys = _keys(row, n, mods, "uniform")
        srv = _shard(_params(n, mods, dim_sum), pb.GaloisKeys(elts, keys), monkeypatch, forced)
        d_q = torch.from_numpy(_queries("uniform", mods, nq, 1, n, seed=3).view(np.int64)).cuda()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            srv.expand_ntt(d_q)
            torch.cuda.synchronize()
        names = set()
        for ev in prof.events():
            m = re.search(r"(k_ks_\w+)(<[^>]*>)?", ev.name)
            if m:
                names.add(m.group(1) + (m.group(2) or "").replace(" ", ""))
        want = _predicted_kernels(n, mods, forced, _level_nodes(n, dim_sum, nq), sms)
        assert names == want, (row, sorted(names), sorted(want))
        for name in names:
            reached.setdefault(_describe(name, n, k), []).append(row)
        del srv, d_q
    with capsys.disabled():
        print("\nkey-switch kernels reached (%d SMs):" % sms)
        for name in sorted(reached):
            print("  %-62s %s" % (name, " ".join(reached[name])))


def test_prediction_reaches_every_instantiation():
    """The rows together reach every key-switch instantiation of interest (prediction for a 148-SM B200)."""
    got = set()
    for row in ROWS:
        n, mods, forced = _row(row)
        got |= _predicted_kernels(n, mods, forced, _level_nodes(n, 40, 5), 148)
    for want in ("k_ks_level_cluster2<11,1>", "k_ks_level_cluster2<11,2>", "k_ks_level_cluster2<12,1>",
                 "k_ks_level_cluster2<12,2>", "k_ks_level_cluster<12,2,2>", "k_ks_level_cluster<11,2,2>",
                 "k_ks_level_cluster<13,2,2>", "k_ks_level_cluster<12,1,1>", "k_ks_level_cluster<12,1,0>",
                 "k_ks_level_cluster<12,0,0>", "k_ks_level_cluster<13,1,1>", "k_ks_level_cluster<13,0,0>",
                 "k_ks_level_cluster<11,0,0>", "k_ks_digits<12,2>", "k_ks_digits<13,2>", "k_ks_digits<14,0>",
                 "k_ks_digits<14,2>", "k_ks_digits<11,2>"):
        assert want in got, want


# ------------------------------------------------------------------------------------------------ order of set-up
_ORDER_SCRIPT = textwrap.dedent("""
    import sys
    sys.path.insert(0, sys.argv[1])
    import numpy as np
    import pir_b200 as pb
    from oracle import binding as ob

    def primes(bits, n, count):
        out, v = [], (1 << bits) - 2 * n + 1
        while len(out) < count:
            if ob.is_prime(v):
                out.append(v)
            v -= 2 * n
        return out

    n = int(sys.argv[2])
    first = primes(30, n, 4) if n == 4096 else primes(44, n, 4)      # k = 3: cluster of 8 CTAs
    second = primes(30, n, 5) if n == 4096 else ob.bfv_default(n)    # k = 4: cluster of 10, same bytes, same kernel
    for mods in (first, second):
        mods = [int(q) for q in mods]
        k = len(mods) - 1
        ep = pb.EncryptionParameters(n, ob.plain_modulus_batching(n, 20), mods)
        p = pb.PIRParameters(num_items=1, num_pt=1, dimensions=[4, 4], encryption_parameters=ep, bytes_per_item=0,
                             items_per_plaintext=1, bits_per_coeff=0)
        db = pb.PIRDatabase(p)
        db.fill_random(1)
        server = pb.PIRServer.Create(db, p)
        rng = np.random.default_rng(k)
        elts = pb.generate_galois_elts(n)
        keys = np.ascontiguousarray(np.stack([rng.integers(0, q, (len(elts), k, 2, n), dtype=np.uint64)
                                              for q in mods], axis=3)).reshape(-1)
        ct = np.ascontiguousarray(np.stack([rng.integers(0, mods[j], (2, n), dtype=np.uint64) for j in range(k)],
                                           axis=1))
        got = server.oblivious_expansion(ct, 8, pb.GaloisKeys(elts, keys))
        want = ob.Oracle(n, mods, ep.plain_modulus).expand(ct, 8, elts, keys, single=True)
        assert np.array_equal(got, want), "k = %d: expansion differs from the oracle" % k
        print("k = %d ok" % k)
""")


@pytest.mark.parametrize("n", [4096, 8192])
def test_cluster_sizes_served_in_either_order(n):
    """A process that first expands with k = 3 (cluster of 8 CTAs) and then with k = 4 (cluster of 10, the same
    dynamic shared memory and the same first-generation instantiation) must configure the kernel for both: 30-bit
    moduli at N = 4096, 44-bit k = 3 and then the default moduli at N = 8192.  A fresh interpreter fixes the order."""
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", _ORDER_SCRIPT, ROOT, str(n)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0 and "k = 4 ok" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]


# ------------------------------------------------------------------------------------------------ default N = 16384
def test_default_n16384_end_to_end(monkeypatch):
    """BFVDefault(16384) (nine moduli of 48/49 bits: corrected integer butterflies, 128-bit MACs, k = 8, three-launch
    expansion) end to end on a d = 2 database with real keys: one query decrypts to its item and its reply equals the
    oracle's limb for limb; a 4-query batch (7 byte limbs per residue: no tensor-core plan, so the CUDA-core 128-bit
    batch scan) answers every query as the single-query path does."""
    monkeypatch.setenv("PIRB_TC_MIN_PT", "0")  # the tensor-core scan may take this batch if it has a plan for it
    ep = pb.GenerateEncryptionParams(16384, 20)
    assert len(ep.coeff_modulus) == 9
    p = pb.CreatePIRParameters(100, 8192, 2, ep)
    hp = oc.PIRParameters(p.num_items, p.num_pt, list(p.dimensions), p.bytes_per_item, p.items_per_plaintext,
                          p.bits_per_coeff, ep.poly_modulus_degree, ep.plain_modulus, list(ep.coeff_modulus))
    cl = oc.HarnessClient(hp, seed=5)
    rng = np.random.default_rng(16384)
    items = [rng.integers(0, 256, p.bytes_per_item, dtype=np.uint8).tobytes() for _ in range(p.num_items)]
    db = pb.PIRDatabase.Create(items, p)
    server = pb.PIRServer.Create(db, p)
    gk = pb.GaloisKeys(cl.elts, cl.galois)
    idx = [63, 0, 99, 17]
    qs = [cl.create_query(i) for i in idx]
    single = [server.ProcessRequest(pb.Request([q], gk)).reply[0] for q in qs]
    want = cl.orc.process_query(oc.db_to_ntt(cl.orc, oc.encode_string_db(hp, items)), p.dimensions, cl.elts,
                                cl.galois, qs[0])
    assert np.array_equal(single[0], want)
    assert cl.process_response_strings([idx[0]], [single[0]])[0] == items[idx[0]]
    batch = server.ProcessRequest(pb.Request(qs, gk)).reply
    for i in range(len(qs)):
        assert np.array_equal(batch[i], single[i]), i
