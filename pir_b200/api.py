"""Host-side mirror of the reference's server interface for the answer path, on top of the C ABI.

Names, argument meaning and error behaviour follow pir/cpp/server.h:43-131, pir/cpp/database.h:47-127 and
pir/cpp/parameters.h:40-75, with SEAL objects replaced by raw RNS limbs (numpy uint64 arrays):

    ciphertext  [2][k][N]      Galois keys  [n_elts][k][2][k+1][N] (NTT form) + the list of Galois elements
    Request     .query = list of [n_ct][2][k][N] arrays, .galois_keys = GaloisKeys
    Response    .reply = list of [reply_cts][2][k][N] arrays

absl::Status codes surface as PIRStatusError(code): 3 = InvalidArgument, 13 = Internal.
"""
import ctypes as C
from collections import OrderedDict
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np

from . import _lib

INVALID_ARGUMENT = 3
INTERNAL = 13
DEFAULT_POLY_MODULUS_DEGREE = 4096  # parameters.h:40


class PIRStatusError(Exception):
    def __init__(self, code, message):
        super().__init__("[%d] %s" % (code, message))
        self.code = code
        self.message = message


def _check(rc):
    if rc:
        raise PIRStatusError(rc, _lib.last_error())


def _u64(a):
    a = np.ascontiguousarray(a, dtype=np.uint64)
    return a


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


# ---------------------------------------------------------------------------------------------------
# shape math (exported by the C library so it has a single implementation)
# ---------------------------------------------------------------------------------------------------
def next_power_two(v):
    return int(_lib.lib().pirb_next_power_two(v))


def ceil_log2(v):
    return int(_lib.lib().pirb_ceil_log2(v))


def log2(v):
    return int(_lib.lib().pirb_log2(v))


def generate_galois_elts(N):
    """utils.cpp:7-14"""
    return [(N >> i) + 1 for i in range(ceil_log2(N))]


def calculate_dimensions(db_size, num_dimensions):
    """PIRDatabase::calculate_dimensions (database.cpp:334-342)"""
    out = (C.c_uint32 * num_dimensions)()
    _lib.lib().pirb_calculate_dimensions(db_size, num_dimensions, out)
    return [int(x) for x in out]


@dataclass
class EncryptionParameters:
    """The part of seal::EncryptionParameters this path needs."""
    poly_modulus_degree: int
    plain_modulus: int
    coeff_modulus: List[int]  # data-level primes followed by the special prime


def GenerateEncryptionParams(poly_modulus_degree=DEFAULT_POLY_MODULUS_DEGREE, plain_mod_bit_size=20,
                             plain_modulus=None, coeff_modulus=None):
    """parameters.cpp:33-54: PlainModulus::Batching(N, bits) and CoeffModulus::BFVDefault(N) unless given."""
    L = _lib.lib()
    if plain_modulus is None:
        plain_modulus = int(L.pirb_plain_modulus_batching(poly_modulus_degree, plain_mod_bit_size))
        if not plain_modulus:
            raise PIRStatusError(INVALID_ARGUMENT, "failed to find enough qualifying primes")
    if coeff_modulus is None:
        buf = (C.c_uint64 * _lib.PIRB_MAX_MODULI)()
        n = L.pirb_bfv_default_coeff_modulus(poly_modulus_degree, buf, _lib.PIRB_MAX_MODULI)
        if n < 0:
            raise PIRStatusError(INVALID_ARGUMENT, "no default coefficient modulus for this degree")
        coeff_modulus = [int(buf[i]) for i in range(n)]
    return EncryptionParameters(poly_modulus_degree, int(plain_modulus), list(coeff_modulus))


@dataclass
class PIRParameters:
    """pir/proto/payload.proto:45-69"""
    num_items: int = 0
    num_pt: int = 0
    dimensions: List[int] = field(default_factory=list)
    encryption_parameters: Optional[EncryptionParameters] = None
    bytes_per_item: int = 0
    items_per_plaintext: int = 0
    bits_per_coeff: int = 0
    use_ciphertext_multiplication: bool = False


def CreatePIRParameters(dbsize, bytes_per_item=0, dimensions=1, seal_params=None,
                        use_ciphertext_multiplication=False, bits_per_coeff=0):
    """parameters.cpp:56-107"""
    if seal_params is None:
        seal_params = GenerateEncryptionParams()
    enc = StringEncoder(seal_params)
    p = PIRParameters(num_items=dbsize, encryption_parameters=seal_params,
                      use_ciphertext_multiplication=bool(use_ciphertext_multiplication))  # parameters.cpp:71
    if bits_per_coeff > 0:
        if bits_per_coeff > enc.bits_per_coeff:
            raise PIRStatusError(INVALID_ARGUMENT, "Bits per coefficient greater than max")
        enc.set_bits_per_coeff(bits_per_coeff)
        p.bits_per_coeff = bits_per_coeff
    if bytes_per_item > 0:
        p.bytes_per_item = bytes_per_item
        p.items_per_plaintext = enc.num_items_per_plaintext(bytes_per_item)
        if p.items_per_plaintext <= 0:
            raise PIRStatusError(INVALID_ARGUMENT, "Cannot fit an item within one plaintext")
        num_pt = dbsize // p.items_per_plaintext
        while dbsize > num_pt * p.items_per_plaintext:
            num_pt += 1
        p.num_pt = num_pt
    else:
        p.bytes_per_item = enc.max_bytes_per_plaintext()
        p.items_per_plaintext = 1
        p.num_pt = dbsize
    p.dimensions = calculate_dimensions(p.num_pt, dimensions)
    return p


class StringEncoder:
    """string_encoder.{h,cpp}: MSB-first packing of bytes into bits_per_coeff-bit coefficients (host side)."""

    def __init__(self, seal_params: EncryptionParameters):
        self.poly_modulus_degree = seal_params.poly_modulus_degree
        # string_encoder.cpp:85: pir::log2 takes a uint32_t, a wider plain modulus is truncated to its low 32 bits
        self.bits_per_coeff = log2(seal_params.plain_modulus & 0xFFFFFFFF)

    def set_bits_per_coeff(self, b):
        self.bits_per_coeff = b

    def num_items_per_plaintext(self, item_size):
        return self.poly_modulus_degree * self.bits_per_coeff // item_size // 8

    def max_bytes_per_plaintext(self):
        return self.poly_modulus_degree * self.bits_per_coeff // 8

    def encode(self, data: bytes):
        """string_encoder.cpp:58-80,95-122 -> coefficient array (length = ceil(8*len/bits))."""
        b = self.bits_per_coeff
        n_coeff = -(-len(data) * 8 // b) if data else 0
        if n_coeff > self.poly_modulus_degree:
            raise PIRStatusError(INVALID_ARGUMENT, "Number of coefficients needed greater than poly modulus degree")
        if not n_coeff:
            return np.zeros(0, dtype=np.uint64)
        bits = np.unpackbits(np.frombuffer(data, dtype=np.uint8))
        pad = n_coeff * b - bits.size
        if pad:
            bits = np.concatenate([bits, np.zeros(pad, dtype=np.uint8)])
        weights = (np.uint64(1) << np.arange(b - 1, -1, -1, dtype=np.uint64))
        return (bits.reshape(n_coeff, b).astype(np.uint64) * weights).sum(axis=1, dtype=np.uint64)

    def decode(self, coeffs, length=0, byte_offset=0):
        """string_encoder.cpp:124-158"""
        b = self.bits_per_coeff
        coeffs = np.asarray(coeffs, dtype=np.uint64)
        if byte_offset + length > coeffs.size * b // 8:
            raise PIRStatusError(INVALID_ARGUMENT, "Requested decode beyond end of data in polynomial")
        if length <= 0:
            nz = np.nonzero(coeffs)[0]
            length = (int(nz[-1]) + 1 if nz.size else 0) * b // 8
        shifts = np.arange(b - 1, -1, -1, dtype=np.uint64)
        bits = ((coeffs[:, None] >> shifts) & np.uint64(1)).astype(np.uint8).reshape(-1)
        seg = bits[byte_offset * 8:(byte_offset + length) * 8]
        return np.packbits(seg).tobytes()


# ---------------------------------------------------------------------------------------------------
class GaloisKeys:
    """seal::GaloisKeys as raw limbs: elts[i] is the Galois element of data[i] ([k][2][k+1][N], NTT form)."""

    def __init__(self, elts: Sequence[int], data):
        self.elts = [int(e) for e in elts]
        self.data = _u64(data)


@dataclass
class Request:
    """payload.proto:28-36"""
    query: List[np.ndarray] = field(default_factory=list)
    galois_keys: Optional[GaloisKeys] = None
    # seal::RelinKeys as raw limbs [k][2][k+1][N] (one key, NTT form).  Used in ciphertext-multiplication mode
    # (server.cpp:185-190); parsed but unused on the re-encoder path (server.cpp:53-58)
    relin_keys: Optional[object] = None


@dataclass
class Response:
    """payload.proto:39-42"""
    reply: List[np.ndarray] = field(default_factory=list)


class _Context:
    """Owns one pirb_ctx (PIRContext + device state)."""

    def __init__(self, params: PIRParameters, device=0, shard_index=0, shard_count=1):
        ep = params.encryption_parameters
        pp = _lib.pirb_params()
        pp.poly_modulus_degree = ep.poly_modulus_degree
        pp.n_moduli = len(ep.coeff_modulus)
        if pp.n_moduli > _lib.PIRB_MAX_MODULI:
            raise PIRStatusError(INVALID_ARGUMENT, "too many coefficient moduli")
        for i, q in enumerate(ep.coeff_modulus):
            pp.coeff_modulus[i] = q
        pp.plain_modulus = ep.plain_modulus
        pp.n_dims = len(params.dimensions)
        if pp.n_dims > _lib.PIRB_MAX_DIMS:
            raise PIRStatusError(INVALID_ARGUMENT, "too many dimensions")
        for i, d in enumerate(params.dimensions):
            pp.dims[i] = d
        pp.num_pt = params.num_pt
        pp.device = device
        pp.shard_index = shard_index
        pp.shard_count = shard_count
        pp.use_ciphertext_multiplication = 1 if params.use_ciphertext_multiplication else 0
        self.ct_mode = bool(params.use_ciphertext_multiplication)
        h = C.c_void_p()
        _check(_lib.lib().pirb_ctx_create(C.byref(pp), C.byref(h)))
        self.h = h
        L = _lib.lib()
        self.N = ep.poly_modulus_degree
        self.k = len(ep.coeff_modulus) - 1
        self.ct_limbs = int(L.pirb_ct_limbs(h))
        self.pt_limbs = int(L.pirb_pt_limbs(h))
        self.key_limbs = int(L.pirb_key_limbs(h))
        self.reply_cts = int(L.pirb_reply_cts(h))
        self.dim_sum = int(L.pirb_dim_sum(h))
        self.query_cts = int(L.pirb_query_cts(h))
        self.expansion_ratio = int(L.pirb_expansion_ratio(h))

    def close(self):
        if getattr(self, "h", None):
            _lib.lib().pirb_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class _KeyHandle:
    def __init__(self, ctx: _Context, gk: GaloisKeys):
        self.h = C.c_void_p()
        elts = (C.c_uint32 * max(1, len(gk.elts)))(*gk.elts)
        if gk.data.size != len(gk.elts) * ctx.key_limbs:
            raise PIRStatusError(INVALID_ARGUMENT, "Galois key data has the wrong size")
        _check(_lib.lib().pirb_keys_load(ctx.h, elts, len(gk.elts), _ptr(gk.data), C.byref(self.h)))

    def close(self):
        if getattr(self, "h", None):
            _lib.lib().pirb_keys_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class _RelinHandle:
    """seal::RelinKeys (one key-switching key for s^2) resident in HBM."""

    def __init__(self, ctx: _Context, limbs):
        self.h = C.c_void_p()
        a = _u64(limbs)
        if a.size != ctx.key_limbs:
            raise PIRStatusError(INVALID_ARGUMENT, "relinearization key data has the wrong size")
        _check(_lib.lib().pirb_relin_keys_load(ctx.h, _ptr(a), C.byref(self.h)))

    def close(self):
        if getattr(self, "h", None):
            _lib.lib().pirb_keys_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class PIRDatabase:
    """database.h:47-127.  The plaintexts live in HBM in NTT form (RNS uint64 limbs)."""

    def __init__(self, params: PIRParameters, device=0, shard_index=0, shard_count=1):
        self.params = params
        self.ctx = _Context(params, device, shard_index, shard_count)

    # -- factories ------------------------------------------------------------------------------
    @classmethod
    def Create(cls, params_or_rawdb, params: PIRParameters = None, **kw):
        """Create(params) | Create(vector<int64>, params) | Create(vector<string>, params) (database.cpp:38-58)"""
        if params is None:
            return cls(params_or_rawdb, **kw)
        db = cls(params, **kw)
        db.populate(params_or_rawdb)
        return db

    def populate(self, rawdb):
        """database.cpp:60-110"""
        p = self.params
        if len(rawdb) != p.num_items:
            raise PIRStatusError(INVALID_ARGUMENT, "Database size %d does not match params value %d" %
                                 (len(rawdb), p.num_items))
        N = p.encryption_parameters.poly_modulus_degree
        if len(rawdb) and isinstance(rawdb[0], (bytes, bytearray, str)) and \
                all(len(x) == p.bytes_per_item for x in rawdb):
            # fixed-size items: ship the raw bytes, pack + lift + NTT on the GPU
            ipp = p.items_per_plaintext
            per_chunk = max(ipp, ((64 << 20) // max(1, p.bytes_per_item)) // ipp * ipp)
            for start in range(0, len(rawdb), per_chunk):
                chunk = rawdb[start:start + per_chunk]
                blob = b"".join(x.encode("latin1") if isinstance(x, str) else bytes(x) for x in chunk)
                self.load_items(blob, start, len(chunk))
        elif len(rawdb) and isinstance(rawdb[0], (bytes, bytearray, str)):
            enc = StringEncoder(p.encryption_parameters)
            if p.bits_per_coeff > 0:
                enc.set_bits_per_coeff(p.bits_per_coeff)
            ipp = p.items_per_plaintext
            chunk = max(1, (32 << 20) // (N * 8))
            for start in range(0, p.num_pt, chunk):
                stop = min(p.num_pt, start + chunk)
                buf = np.zeros((stop - start, N), dtype=np.uint64)
                for i in range(start, stop):
                    items = rawdb[i * ipp:(i + 1) * ipp]
                    blob = b"".join(x.encode("latin1") if isinstance(x, str) else bytes(x) for x in items)
                    c = enc.encode(blob)
                    buf[i - start, :c.size] = c
                self.load_coeff(buf, start)
        else:
            if p.num_pt != p.num_items:
                raise PIRStatusError(INVALID_ARGUMENT, "integer database needs one item per plaintext")
            t = p.encryption_parameters.plain_modulus
            buf = np.zeros((len(rawdb), N), dtype=np.uint64)
            for i, v in enumerate(rawdb):
                buf[i] = integer_encode(int(v), N, t)
            self.load_coeff(buf, 0)

    def load_coeff(self, coeffs, first_pt=0):
        a = _u64(coeffs).reshape(-1, self.ctx.N)
        _check(_lib.lib().pirb_db_load_coeff(self.ctx.h, _ptr(a), first_pt, a.shape[0]))

    def load_items(self, blob: bytes, first_item: int, n_items: int):
        """Raw fixed-size items -> packed, lifted, NTT-transformed on the device (pirb_db_load_items)."""
        p = self.params
        buf = np.frombuffer(blob, dtype=np.uint8)
        _check(_lib.lib().pirb_db_load_items(self.ctx.h, _ptr(buf), first_item, n_items, p.bytes_per_item,
                                             p.items_per_plaintext, p.bits_per_coeff))

    def save(self, path: str, chunk_pt: int = 4096):
        """Persist this shard's preprocessed (NTT-form) plaintexts: 64-byte header + raw little-endian u64 limbs."""
        L = _lib.lib()
        begin, count = int(L.pirb_shard_pt_begin(self.ctx.h)), int(L.pirb_shard_pt_count(self.ctx.h))
        hdr = np.zeros(8, dtype=np.uint64)
        hdr[:6] = [0x3142444252495042, self.ctx.N, self.ctx.k, begin, count, self.params.encryption_parameters.plain_modulus]
        with open(path, "wb") as f:
            f.write(hdr.tobytes())
            f.write(np.array(self.params.encryption_parameters.coeff_modulus, dtype=np.uint64).tobytes())
            for s0 in range(begin, begin + count, chunk_pt):
                n = min(chunk_pt, begin + count - s0)
                f.write(self.read_ntt(s0, n).tobytes())

    def load(self, path: str, chunk_pt: int = 4096):
        """Load a shard file written by save(); the parameters must match."""
        ep = self.params.encryption_parameters
        with open(path, "rb") as f:
            hdr = np.frombuffer(f.read(64), dtype=np.uint64)
            mods = np.frombuffer(f.read(8 * len(ep.coeff_modulus)), dtype=np.uint64)
            if int(hdr[0]) != 0x3142444252495042 or int(hdr[1]) != self.ctx.N or int(hdr[2]) != self.ctx.k or \
                    int(hdr[5]) != ep.plain_modulus or [int(x) for x in mods] != list(ep.coeff_modulus):
                raise PIRStatusError(INVALID_ARGUMENT, "shard file does not match the parameters")
            begin, count = int(hdr[3]), int(hdr[4])
            for s0 in range(begin, begin + count, chunk_pt):
                n = min(chunk_pt, begin + count - s0)
                a = np.frombuffer(f.read(n * self.ctx.pt_limbs * 8), dtype=np.uint64)
                self.load_ntt(a, s0)

    def load_ntt(self, limbs, first_pt=0):
        a = _u64(limbs).reshape(-1, self.ctx.pt_limbs)
        _check(_lib.lib().pirb_db_load_ntt(self.ctx.h, _ptr(a), first_pt, a.shape[0]))

    def read_ntt(self, first_pt, count):
        out = np.zeros((count, self.ctx.k, self.ctx.N), dtype=np.uint64)
        _check(_lib.lib().pirb_db_read_ntt(self.ctx.h, _ptr(out), first_pt, count))
        return out

    def fill_random(self, seed=42):
        _check(_lib.lib().pirb_db_fill_random(self.ctx.h, seed))

    def size(self):
        """database.h:94 — number of plaintexts held"""
        return int(_lib.lib().pirb_db_size(self.ctx.h))

    # -- the hot path ---------------------------------------------------------------------------
    def multiply(self, selection_vector: np.ndarray, relin_keys=None, decryptor=None):
        """database.cpp:290-316.  selection_vector [dim_sum][2][k][N] is mutated to NTT form in place."""
        sv = selection_vector
        if sv.dtype != np.uint64 or not sv.flags["C_CONTIGUOUS"]:
            raise PIRStatusError(INVALID_ARGUMENT, "selection vector must be a C-contiguous uint64 array")
        n_sv = sv.size // self.ctx.ct_limbs
        if self.ctx.ct_mode:
            # database.cpp:202-211: Evaluator::multiply (+ relinearize_inplace when keys are given); the selection
            # vector stays in coefficient form; ONE result ciphertext [polys][k][N]
            rh = _RelinHandle(self.ctx, relin_keys) if relin_keys is not None else None
            try:
                polys = int(_lib.lib().pirb_reply_polys(self.ctx.h, 1 if rh else 0))
                out = np.zeros((polys, self.ctx.k, self.ctx.N), dtype=np.uint64)
                got = C.c_uint32(0)
                _check(_lib.lib().pirb_db_multiply_ct(self.ctx.h, _ptr(sv), n_sv, rh.h if rh else None, _ptr(out), out.size,
                                                      C.byref(got)))
            finally:
                if rh:
                    rh.close()
            return out[None] if got.value else out[:0][None]
        out = np.zeros((self.ctx.reply_cts, 2, self.ctx.k, self.ctx.N), dtype=np.uint64)
        cnt = C.c_uint64(0)
        _check(_lib.lib().pirb_db_multiply(self.ctx.h, _ptr(sv), n_sv, _ptr(out), out.shape[0], C.byref(cnt)))
        return out[:cnt.value]

    # -- index math (database.cpp:318-332) ------------------------------------------------------
    def calculate_indices(self, index):
        p = self.params
        pt_index = index // p.items_per_plaintext
        res = [0] * len(p.dimensions)
        for i in range(len(res) - 1, -1, -1):
            res[i] = pt_index % p.dimensions[i]
            pt_index //= p.dimensions[i]
        return res

    def calculate_item_offset(self, index):
        p = self.params
        pt_index = index // p.items_per_plaintext
        return (index - pt_index * p.items_per_plaintext) * p.bytes_per_item

    calculate_dimensions = staticmethod(calculate_dimensions)


def integer_encode(value, N, t):
    """SEAL IntegerEncoder::encode(int64) as used by populate(vector<int64>) (database.cpp:69)."""
    pt = np.zeros(N, dtype=np.uint64)
    neg = value < 0
    v = -value if neg else value
    i = 0
    while v:
        if v & 1:
            pt[i] = (t - 1) if neg else 1
        v >>= 1
        i += 1
    return pt


class PIRServer:
    """server.h:43-131"""

    def __init__(self, db: PIRDatabase, params: PIRParameters):
        self.db_ = db
        self.params = params
        self.ctx = db.ctx  # device state is shared with the database it serves
        self._key_cache = (None, None)
        self._relin_cache = (None, None)
        # ProcessRequests: key handles of recent clients, least recently used first, keyed on the GaloisKeys object
        self.key_cache_capacity = 16
        self._multi_key_cache = OrderedDict()  # id(GaloisKeys) -> (GaloisKeys, _KeyHandle)

    @classmethod
    def Create(cls, db: PIRDatabase, params: PIRParameters):
        if params.num_pt != db.size():  # server.cpp:37-39
            raise PIRStatusError(INVALID_ARGUMENT, "database size mismatch")
        return cls(db, params)

    def _keys(self, gk: GaloisKeys):
        if gk is None:
            raise PIRStatusError(INVALID_ARGUMENT, "galois keys missing")  # SEALDeserialize failure, serialization.h:113-115
        if self._key_cache[0] is not gk:
            old = self._key_cache[1]
            self._key_cache = (gk, _KeyHandle(self.ctx, gk))
            if old is not None:
                old.close()
        return self._key_cache[1]

    def ProcessRequest(self, request: Request, out: np.ndarray = None) -> Response:
        """server.cpp:44-65: every query of the request, in order, with the request's Galois keys.
        `out` (optional, extension): caller-provided [n_queries][reply_cts][2][k][N] uint64 buffer (e.g. pinned)."""
        keys = self._keys(request.galois_keys)
        resp = Response()
        if not request.query:
            return resp
        n_q = len(request.query)
        n_ct = request.query[0].size // self.ctx.ct_limbs
        same = all(q.size // self.ctx.ct_limbs == n_ct for q in request.query)
        if not same or n_ct != self.ctx.query_cts:
            raise PIRStatusError(INVALID_ARGUMENT,
                                 "Number of ciphertexts doesn't match number of items for oblivious expansion.")
        if n_q == 1:
            q = _u64(request.query[0])  # no copy when already contiguous uint64
        else:
            q = _u64(np.stack([np.asarray(x).reshape(n_ct, 2, self.ctx.k, self.ctx.N) for x in request.query]))
        if getattr(self.ctx, "ct_mode", False):
            # server.cpp:185-190: relinearization keys, when the request carries them, are applied after every
            # ciphertext multiplication; each reply is ONE ciphertext of `polys` polynomials (client.cpp:196-217)
            rk = request.relin_keys
            if rk is not None and self._relin_cache[0] is not rk:
                old = self._relin_cache[1]
                self._relin_cache = (rk, _RelinHandle(self.ctx, rk))
                if old is not None:
                    old.close()
            rh = self._relin_cache[1] if rk is not None else None
            polys = int(_lib.lib().pirb_reply_polys(self.ctx.h, 1 if rh else 0))
            res = np.empty((n_q, 1, polys, self.ctx.k, self.ctx.N), dtype=np.uint64)
            _check(_lib.lib().pirb_answer_ct(self.ctx.h, keys.h, rh.h if rh else None, C.c_void_p(q.ctypes.data), n_q, n_ct,
                                             C.c_void_p(res.ctypes.data)))
            resp.reply = [res[i] for i in range(n_q)]
            return resp
        shape = (n_q, self.ctx.reply_cts, 2, self.ctx.k, self.ctx.N)
        if out is None:
            out = np.empty(shape, dtype=np.uint64)
        elif out.dtype != np.uint64 or out.size != n_q * self.ctx.reply_cts * self.ctx.ct_limbs or \
                not out.flags["C_CONTIGUOUS"]:
            raise PIRStatusError(INVALID_ARGUMENT, "bad output buffer")
        # q and out are locals that outlive the call, so plain addresses are enough (ndarray.ctypes.data_as costs 4 us)
        _check(_lib.lib().pirb_answer(self.ctx.h, keys.h, C.c_void_p(q.ctypes.data), n_q, n_ct,
                                      C.c_void_p(out.ctypes.data)))
        out = out.reshape(shape)
        resp.reply = [out[i] for i in range(n_q)]
        return resp

    def _trim_key_cache(self, keep=()):
        """Close the least recently used handles beyond key_cache_capacity, except those in `keep`: closing a handle
        frees its keys on the device, so the handles of a batch stay open until its call has returned."""
        over = len(self._multi_key_cache) - max(1, int(self.key_cache_capacity))
        for key in list(self._multi_key_cache):
            if over <= 0:
                break
            if key not in keep:
                self._multi_key_cache.pop(key)[1].close()
                over -= 1

    def _batch_keys(self, gks):
        """One handle per GaloisKeys object of the batch (cached across calls), in batch order."""
        handles, used = [], set()
        for gk in gks:
            key = id(gk)  # the cache holds the object, so its id is not reused while the entry lives
            if key in self._multi_key_cache:
                self._multi_key_cache.move_to_end(key)
            else:
                self._multi_key_cache[key] = (gk, _KeyHandle(self.ctx, gk))
            used.add(key)
            self._trim_key_cache(keep=used)
            handles.append(self._multi_key_cache[key][1])
        return handles

    def ProcessRequests(self, requests: List[Request]) -> List[Response]:
        """ProcessRequest for requests of several clients, each with its own Galois keys, in one batched device call
        (pirb_answer_multi): the Response of each request equals what ProcessRequest returns for it alone.  Key handles
        come from an LRU of key_cache_capacity clients keyed on the GaloisKeys object.  In ciphertext-multiplication
        mode the requests are answered one by one."""
        requests = list(requests)
        for r in requests:
            if r.galois_keys is None:
                raise PIRStatusError(INVALID_ARGUMENT, "galois keys missing")
        if getattr(self.ctx, "ct_mode", False):
            return [self.ProcessRequest(r) for r in requests]
        n_ct = self.ctx.query_cts
        for r in requests:
            if any(q.size // self.ctx.ct_limbs != n_ct for q in r.query):
                raise PIRStatusError(INVALID_ARGUMENT,
                                     "Number of ciphertexts doesn't match number of items for oblivious expansion.")
        shape = (n_ct, 2, self.ctx.k, self.ctx.N)
        queries = [np.asarray(q).reshape(shape) for r in requests for q in r.query]
        owners = [r.galois_keys for r in requests for _ in r.query]
        n_q = len(queries)
        if not n_q:
            return [Response() for _ in requests]
        q = _u64(np.stack(queries))
        out = np.empty((n_q, self.ctx.reply_cts, 2, self.ctx.k, self.ctx.N), dtype=np.uint64)
        try:
            handles = self._batch_keys(owners)
            table = (C.c_void_p * n_q)(*[h.h.value for h in handles])
            _check(_lib.lib().pirb_answer_multi(self.ctx.h, table, C.c_void_p(q.ctypes.data), n_q, n_ct,
                                                C.c_void_p(out.ctypes.data)))
        finally:
            self._trim_key_cache()
        res, i = [], 0
        for r in requests:
            res.append(Response(reply=[out[i + j] for j in range(len(r.query))]))
            i += len(r.query)
        return res

    def ProcessRequestBytes(self, serialized_request: bytes) -> bytes:
        """server.cpp:44-65 on the wire: a serialized pir.Request (protobuf framing, SEAL 3.5.6 objects, seed-compressed
        keys included) in, a serialized pir.Response out.  InvalidArgument on any deserialization failure
        (serialization.h:113-115).  The codec is host-side (pir_b200/wire.py); the answer is ProcessRequest's."""
        from . import wire
        request = wire.parse_request(serialized_request, self.params)
        return wire.serialize_response(self.ProcessRequest(request), self.params, parms_id=request.parms_id)

    def substitute_power_x_inplace(self, ct: np.ndarray, power: int, gal_keys: GaloisKeys):
        """server.cpp:67-76"""
        keys = self._keys(gal_keys)
        _check(_lib.lib().pirb_substitute(self.ctx.h, keys.h, _ptr(ct), power))

    def multiply_inverse_power_of_x(self, encrypted: np.ndarray, k: int):
        """server.cpp:78-103 (returns the destination)"""
        a = _u64(encrypted)
        out = np.zeros_like(a)
        _check(_lib.lib().pirb_mul_inv_pow_x(self.ctx.h, _ptr(a), k, _ptr(out)))
        return out

    def oblivious_expansion(self, ct_or_cts: np.ndarray, num_items: int, gal_keys: GaloisKeys):
        """server.cpp:105-146 for one ciphertext ([2][k][N]), server.cpp:148-171 for several ([n][2][k][N])."""
        keys = self._keys(gal_keys)
        a = _u64(ct_or_cts)
        single = a.ndim == 3
        n_ct = 1 if single else a.shape[0]
        out = np.zeros((num_items, 2, self.ctx.k, self.ctx.N), dtype=np.uint64)
        _check(_lib.lib().pirb_expand(self.ctx.h, keys.h, _ptr(a), n_ct, num_items, 1 if single else 0, _ptr(out)))
        return out

    def Context(self):
        return self.ctx
