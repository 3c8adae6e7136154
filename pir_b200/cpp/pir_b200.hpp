// pir_b200.hpp — C++17 host-side mirror of the reference's server interface over the C ABI (include/pir_b200.h).
//
// Same class names, method names, argument meaning and status codes as OpenMined/PIR's pir::PIRServer
// (pir/cpp/server.h:43-131), pir::PIRDatabase (pir/cpp/database.h:47-127), CreatePIRParameters
// (pir/cpp/parameters.h:55-73) and StringEncoder (pir/cpp/string_encoder.h), with SEAL / abseil / protobuf types
// replaced by plain structs of raw RNS limbs (those libraries are not available in this image):
//
//   pir::Ciphertext   std::vector<uint64_t> limbs, layout [2][k][N]  == seal::Ciphertext::data()
//   pir::GaloisKeys   elts[i] + limbs [n][k][2][k+1][N]               == seal::GaloisKeys (KSwitchKeys layout)
//   pir::Request      { query: vector<vector<Ciphertext>>, galois_keys }   (payload.proto:28-36)
//   pir::Response     { reply: vector<vector<Ciphertext>> }                (payload.proto:39-42)
//   pir::Status / StatusOr<T>   codes as absl::StatusCode: 0 OK, 3 InvalidArgument, 13 Internal
//
// The reference's wire format is layered on top (wire.hpp): PIRServer::ProcessRequest(const std::string&) takes a
// serialized pir.Request (protobuf framing + SEAL 3.5.6 objects, seed-compressed keys included) and returns a
// serialized pir.Response; SerializePIRParameters / ParsePIRParameters do the same for pir.PIRParameters.
//
// Header-only; link with -lpirb200.  All ring arithmetic runs in the CUDA kernels behind the C ABI; nothing here
// computes on ciphertexts.
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <memory>
#include <numeric>
#include <optional>
#include <string>
#include <utility>
#include <vector>

#include "../../include/pir_b200.h"
#include "wire.hpp"

namespace pir {

// ---------------------------------------------------------------------------------------------------------------
struct Status {
  int code_ = 0;
  std::string message_;
  Status() {}
  Status(int c, std::string m) : code_(c), message_(std::move(m)) {}
  bool ok() const { return code_ == 0; }
  int code() const { return code_; }
  const std::string& message() const { return message_; }
};
inline Status OkStatus() { return Status(); }
inline Status InvalidArgumentError(const std::string& m) { return Status(PIRB_INVALID_ARGUMENT, m); }
inline Status InternalError(const std::string& m) { return Status(PIRB_INTERNAL, m); }
inline Status FromRc(int rc) { return rc ? Status(rc, pirb_last_error()) : Status(); }

template <typename T>
class StatusOr {
 public:
  StatusOr(const Status& s) : status_(s) {}          // NOLINT
  StatusOr(T v) : value_(std::move(v)) {}            // NOLINT
  bool ok() const { return status_.ok(); }
  const Status& status() const { return status_; }
  T& value() { return *value_; }
  const T& value() const { return *value_; }
  T& operator*() { return *value_; }
  T* operator->() { return &*value_; }

 private:
  Status status_;
  std::optional<T> value_;
};

// ---------------------------------------------------------------------------------------------------------------
constexpr uint32_t DEFAULT_POLY_MODULUS_DEGREE = 4096;  // parameters.h:40

struct EncryptionParameters {
  uint32_t poly_modulus_degree = 0;
  uint64_t plain_modulus = 0;
  std::vector<uint64_t> coeff_modulus;  // data primes, then the special prime
};

// parameters.cpp:33-54
inline EncryptionParameters GenerateEncryptionParams(uint32_t poly_mod_degree = DEFAULT_POLY_MODULUS_DEGREE,
                                                     uint32_t plain_mod_bit_size = 20) {
  EncryptionParameters p;
  p.poly_modulus_degree = poly_mod_degree;
  p.plain_modulus = pirb_plain_modulus_batching(poly_mod_degree, plain_mod_bit_size);
  uint64_t buf[PIRB_MAX_MODULI];
  int n = pirb_bfv_default_coeff_modulus(poly_mod_degree, buf, PIRB_MAX_MODULI);
  if (n > 0) p.coeff_modulus.assign(buf, buf + n);
  return p;
}

// pir/proto/payload.proto:45-69
struct PIRParameters {
  uint64_t num_items = 0;
  uint64_t num_pt = 0;
  std::vector<uint32_t> dimensions;
  EncryptionParameters encryption_parameters;
  uint32_t bytes_per_item = 0;
  uint32_t items_per_plaintext = 0;
  uint32_t bits_per_coeff = 0;
  bool use_ciphertext_multiplication = false;
};

// string_encoder.{h,cpp}: MSB-first packing of bytes into bits_per_coeff-bit coefficients
class StringEncoder {
 public:
  explicit StringEncoder(const EncryptionParameters& ep)
      : poly_modulus_degree_(ep.poly_modulus_degree), bits_per_coeff_(pirb_log2((uint32_t)ep.plain_modulus)) {}
  size_t bits_per_coeff() const { return bits_per_coeff_; }
  void set_bits_per_coeff(size_t b) { bits_per_coeff_ = b; }
  size_t num_items_per_plaintext(size_t item_size) const { return poly_modulus_degree_ * bits_per_coeff_ / item_size / 8; }
  size_t max_bytes_per_plaintext() const { return poly_modulus_degree_ * bits_per_coeff_ / 8; }

  // string_encoder.cpp:58-80, 95-122: coefficients of the concatenation of [begin, end)
  Status encode(std::vector<std::string>::const_iterator v, std::vector<std::string>::const_iterator end,
                std::vector<uint64_t>& destination) const {
    size_t total = 0;
    for (auto it = v; it != end; ++it) total += it->size();
    const size_t num_coeff = (size_t)std::ceil(static_cast<double>(total * 8) / bits_per_coeff_);
    if (num_coeff > poly_modulus_degree_)
      return InvalidArgumentError("Number of coefficients needed greater than poly modulus degree");
    destination.assign(num_coeff, 0);
    size_t ci = 0, cb = bits_per_coeff_;
    for (; v != end; ++v)
      for (uint8_t ch : *v) {
        size_t remain = 8;
        while (remain > 0) {
          const size_t n = std::min(cb, remain);
          destination[ci] = (destination[ci] << n) | (uint64_t)(ch >> (8 - n));
          ch = (uint8_t)(ch << n);
          cb -= n;
          remain -= n;
          if (cb == 0) { ++ci; cb = bits_per_coeff_; }
        }
      }
    if (cb < bits_per_coeff_ && cb > 0) destination[ci] <<= cb;
    return OkStatus();
  }
  Status encode(const std::string& value, std::vector<uint64_t>& destination) const {
    std::vector<std::string> one{value};
    return encode(one.cbegin(), one.cend(), destination);
  }
  // string_encoder.cpp:124-158
  StatusOr<std::string> decode(const std::vector<uint64_t>& pt, size_t length, size_t byte_offset = 0) const {
    if ((byte_offset + length) > (pt.size() * bits_per_coeff_ / 8))
      return InvalidArgumentError("Requested decode beyond end of data in polynomial");
    const size_t start = byte_offset * 8 / bits_per_coeff_;
    size_t cb = ((start + 1) * bits_per_coeff_) - (byte_offset * 8);
    if (cb == 0) cb = bits_per_coeff_;
    std::string result(length, 0);
    if (!length) return result;
    size_t ri = 0, remain = 8;
    for (size_t i = start; i < pt.size(); ++i) {
      while (cb > 0) {
        const size_t n = std::min(cb, remain);
        result[ri] = (char)(((uint8_t)result[ri] << n) | (uint8_t)((pt[i] >> (cb - n)) & ((1u << n) - 1)));
        cb -= n;
        remain -= n;
        if (remain == 0) {
          if (++ri >= length) return result;
          remain = 8;
        }
      }
      cb = bits_per_coeff_;
    }
    return result;
  }

 private:
  size_t poly_modulus_degree_;
  size_t bits_per_coeff_;
};

// parameters.cpp:56-107
inline StatusOr<std::shared_ptr<PIRParameters>> CreatePIRParameters(
    size_t dbsize, size_t bytes_per_item = 0, size_t dimensions = 1,
    EncryptionParameters seal_params = GenerateEncryptionParams(), bool use_ciphertext_multiplication = false,
    size_t bits_per_coeff = 0) {
  if (seal_params.coeff_modulus.size() < 2 || !seal_params.plain_modulus)
    return InvalidArgumentError("Error setting encryption parameters: invalid parameters");
  StringEncoder encoder(seal_params);
  auto p = std::make_shared<PIRParameters>();
  p->use_ciphertext_multiplication = use_ciphertext_multiplication;  // parameters.cpp:71
  p->num_items = dbsize;
  p->encryption_parameters = seal_params;
  if (bits_per_coeff > 0) {
    if (bits_per_coeff > encoder.bits_per_coeff()) return InvalidArgumentError("Bits per coefficient greater than max");
    encoder.set_bits_per_coeff(bits_per_coeff);
    p->bits_per_coeff = (uint32_t)bits_per_coeff;
  }
  if (bytes_per_item > 0) {
    p->bytes_per_item = (uint32_t)bytes_per_item;
    p->items_per_plaintext = (uint32_t)encoder.num_items_per_plaintext(bytes_per_item);
    if (p->items_per_plaintext <= 0) return InvalidArgumentError("Cannot fit an item within one plaintext");
    size_t num_pt = dbsize / p->items_per_plaintext;
    while (dbsize > num_pt * p->items_per_plaintext) ++num_pt;
    p->num_pt = num_pt;
  } else {
    p->bytes_per_item = (uint32_t)encoder.max_bytes_per_plaintext();
    p->items_per_plaintext = 1;
    p->num_pt = dbsize;
  }
  p->dimensions.resize(dimensions);
  pirb_calculate_dimensions((uint32_t)p->num_pt, (uint32_t)dimensions, p->dimensions.data());
  return p;
}

// ---------------------------------------------------------------------------------------------------------------
struct Ciphertext {
  std::vector<uint64_t> limbs;  // [2][k][N]  ([size][k][N]: replies of the ciphertext-multiplication mode without
                                // relinearization keys keep more than two polynomials, server.cpp:185-190)
  bool is_ntt_form = false;
  uint64_t* data() { return limbs.data(); }
  const uint64_t* data() const { return limbs.data(); }
};
struct GaloisKeys {
  std::vector<uint32_t> elts;
  std::vector<uint64_t> limbs;  // [n][k][2][k+1][N], NTT form
};
struct RelinKeys {
  std::vector<uint64_t> limbs;  // [k][2][k+1][N], NTT form: the one key KeyGenerator::relin_keys() makes (client.cpp:49)
};
struct Request {
  std::vector<std::vector<Ciphertext>> query;
  GaloisKeys galois_keys;
  std::optional<RelinKeys> relin_keys;  // used in ciphertext-multiplication mode only (server.cpp:53-58, 185-190)
};
struct Response {
  std::vector<std::vector<Ciphertext>> reply;
};

// utils.cpp:7-14
inline std::vector<uint32_t> generate_galois_elts(uint64_t N) {
  std::vector<uint32_t> e(pirb_ceil_log2((uint32_t)N));
  for (size_t i = 0; i < e.size(); ++i) e[i] = (uint32_t)((N >> i) + 1);
  return e;
}

// ---------------------------------------------------------------------------------------------------------------
// wire format (pir/cpp/serialization.h:81-138, pir/proto/payload.proto, parameters.cpp:100-101)
inline wire::SealParams ToSealParams(const EncryptionParameters& ep) {
  wire::SealParams p;
  p.poly_modulus_degree = ep.poly_modulus_degree;
  p.coeff_modulus = ep.coeff_modulus;
  p.plain_modulus = ep.plain_modulus;
  return p;
}
inline std::string SerializePIRParameters(const PIRParameters& p) {
  wire::PIRParametersMsg m;
  m.num_items = p.num_items;
  m.num_pt = p.num_pt;
  m.dimensions = p.dimensions;
  m.encryption_parameters = wire::SaveEncryptionParameters(ToSealParams(p.encryption_parameters));
  m.bytes_per_item = p.bytes_per_item;
  m.items_per_plaintext = p.items_per_plaintext;
  m.bits_per_coeff = p.bits_per_coeff;
  m.use_ciphertext_multiplication = p.use_ciphertext_multiplication;
  return wire::Serialize(m);
}
inline StatusOr<std::shared_ptr<PIRParameters>> ParsePIRParameters(const std::string& bytes) {
  wire::PIRParametersMsg m;
  if (!wire::Parse(bytes, &m)) return InvalidArgumentError("malformed PIRParameters message");
  wire::SealParams sp;
  std::string err;
  if (!wire::LoadEncryptionParameters(m.encryption_parameters, &sp, &err)) return InvalidArgumentError(err);
  auto p = std::make_shared<PIRParameters>();
  p->num_items = m.num_items;
  p->num_pt = m.num_pt;
  p->dimensions = m.dimensions;
  p->encryption_parameters.poly_modulus_degree = sp.poly_modulus_degree;
  p->encryption_parameters.coeff_modulus = sp.coeff_modulus;
  p->encryption_parameters.plain_modulus = sp.plain_modulus;
  p->bytes_per_item = m.bytes_per_item;
  p->items_per_plaintext = m.items_per_plaintext;
  p->bits_per_coeff = m.bits_per_coeff;
  p->use_ciphertext_multiplication = m.use_ciphertext_multiplication;
  return p;
}
// SEALDeserialize<GaloisKeys> (serialization.h:106-121) into the raw-limb key layout of the C ABI
inline StatusOr<GaloisKeys> DeserializeGaloisKeys(const EncryptionParameters& ep, const std::string& bytes) {
  wire::KSwitchKeysData K;
  std::string err;
  if (!wire::LoadKSwitchKeys(bytes, ToSealParams(ep), &K, &err)) return InvalidArgumentError(err);
  GaloisKeys gk;
  const size_t per_digit = 2 * ep.coeff_modulus.size() * (size_t)ep.poly_modulus_degree;
  for (size_t s = 0; s < K.keys.size(); ++s) {
    if (K.keys[s].empty()) continue;
    gk.elts.push_back(wire::galois_elt_of_index((uint32_t)s));
    for (const auto& ct : K.keys[s]) gk.limbs.insert(gk.limbs.end(), ct.limbs.begin(), ct.limbs.begin() + per_digit);
  }
  return gk;
}
inline std::string SerializeGaloisKeys(const EncryptionParameters& ep, const GaloisKeys& gk) {
  const wire::SealParams sp = ToSealParams(ep);
  const size_t N = ep.poly_modulus_degree, k = ep.coeff_modulus.size() - 1, per_digit = 2 * (k + 1) * N;
  wire::KSwitchKeysData K;
  K.parms_id = wire::key_parms_id(sp);
  K.keys.assign(N, {});
  for (size_t e = 0; e < gk.elts.size(); ++e) {
    auto& slot = K.keys[wire::galois_index(gk.elts[e])];
    slot.resize(k);
    for (size_t j = 0; j < k; ++j) {
      slot[j].parms_id = K.parms_id;
      slot[j].is_ntt_form = true;
      slot[j].size = 2;
      slot[j].poly_modulus_degree = N;
      slot[j].coeff_modulus_size = k + 1;
      slot[j].limbs.assign(gk.limbs.begin() + (e * k + j) * per_digit, gk.limbs.begin() + (e * k + j + 1) * per_digit);
    }
  }
  return wire::SaveKSwitchKeys(K);
}
// SEALSerialize<RelinKeys> / SEALDeserialize<RelinKeys>: a KSwitchKeys object with ONE slot (RelinKeys::get_index(2) == 0)
// holding the k digits of the key KeyGenerator::relin_keys() makes (client.cpp:49)
inline std::string SerializeRelinKeys(const EncryptionParameters& ep, const RelinKeys& rk) {
  const wire::SealParams sp = ToSealParams(ep);
  const size_t N = ep.poly_modulus_degree, k = ep.coeff_modulus.size() - 1, per_digit = 2 * (k + 1) * N;
  wire::KSwitchKeysData K;
  K.parms_id = wire::key_parms_id(sp);
  K.keys.resize(1);
  K.keys[0].resize(rk.limbs.size() / per_digit);
  for (size_t j = 0; j < K.keys[0].size(); ++j) {
    auto& c = K.keys[0][j];
    c.parms_id = K.parms_id;
    c.is_ntt_form = true;
    c.size = 2;
    c.poly_modulus_degree = N;
    c.coeff_modulus_size = k + 1;
    c.limbs.assign(rk.limbs.begin() + j * per_digit, rk.limbs.begin() + (j + 1) * per_digit);
  }
  return wire::SaveKSwitchKeys(K);
}
inline StatusOr<RelinKeys> DeserializeRelinKeys(const EncryptionParameters& ep, const std::string& bytes) {
  wire::KSwitchKeysData K;
  std::string err;
  if (!wire::LoadKSwitchKeys(bytes, ToSealParams(ep), &K, &err)) return InvalidArgumentError(err);
  const size_t k = ep.coeff_modulus.size() - 1;
  if (K.keys.size() != 1 || K.keys[0].size() != k)
    return InvalidArgumentError("relinearization keys must hold exactly one key of k digits");
  const size_t per_digit = 2 * ep.coeff_modulus.size() * (size_t)ep.poly_modulus_degree;
  RelinKeys rk;
  for (const auto& ct : K.keys[0]) rk.limbs.insert(rk.limbs.end(), ct.limbs.begin(), ct.limbs.begin() + per_digit);
  return rk;
}
// SEALSerialize<Ciphertext> / SEALDeserialize<Ciphertext> for data-level ciphertexts [2][k][N]
inline std::string SerializeCiphertext(const EncryptionParameters& ep, const Ciphertext& ct,
                                       const wire::parms_id_type* parms_id = nullptr) {
  const wire::SealParams sp = ToSealParams(ep);
  wire::CiphertextData d;
  d.parms_id = parms_id ? *parms_id : wire::data_parms_id(sp);
  d.is_ntt_form = ct.is_ntt_form;
  d.poly_modulus_degree = ep.poly_modulus_degree;
  d.coeff_modulus_size = ep.coeff_modulus.size() - 1;
  d.size = ct.limbs.size() / (d.poly_modulus_degree * d.coeff_modulus_size);
  d.limbs = ct.limbs;
  return wire::SaveCiphertext(d);
}
inline StatusOr<Ciphertext> DeserializeCiphertext(const EncryptionParameters& ep, const std::string& bytes,
                                                  wire::parms_id_type* parms_id = nullptr) {
  wire::CiphertextData d;
  std::string err;
  if (!wire::LoadCiphertext(bytes, ep.poly_modulus_degree, ep.coeff_modulus.data(), ep.coeff_modulus.size() - 1, &d,
                            &err))
    return InvalidArgumentError(err);
  if (d.size != 2) return InvalidArgumentError("ciphertext data is invalid");
  if (parms_id) *parms_id = d.parms_id;
  Ciphertext ct;
  ct.limbs = std::move(d.limbs);
  ct.is_ntt_form = d.is_ntt_form;
  return ct;
}

// serialization.cpp:32-58: Ciphertexts message <-> vector<Ciphertext>
inline StatusOr<std::vector<Ciphertext>> LoadCiphertexts(const EncryptionParameters& ep, const wire::CiphertextsMsg& input) {
  std::vector<Ciphertext> out;
  out.reserve(input.ct.size());
  for (const auto& blob : input.ct) {
    auto ct = DeserializeCiphertext(ep, blob);
    if (!ct.ok()) return ct.status();
    out.push_back(std::move(*ct));
  }
  return out;
}
inline Status SaveCiphertexts(const EncryptionParameters& ep, const std::vector<Ciphertext>& cts, wire::CiphertextsMsg* output) {
  if (output == nullptr) return InvalidArgumentError("output nullptr");
  for (const auto& ct : cts) output->ct.push_back(SerializeCiphertext(ep, ct));
  return OkStatus();
}
// serialization.cpp:53-73: SaveRequest(cts) leaves both key fields empty, SaveRequest(cts, galois, relin) fills them
inline Status SaveRequest(const EncryptionParameters& ep, const std::vector<std::vector<Ciphertext>>& cts,
                          wire::RequestMsg* request) {
  if (request == nullptr) return InvalidArgumentError("output nullptr");
  for (const auto& q : cts) {
    request->query.emplace_back();
    Status st = SaveCiphertexts(ep, q, &request->query.back());
    if (!st.ok()) return st;
  }
  return OkStatus();
}
inline Status SaveRequest(const EncryptionParameters& ep, const std::vector<std::vector<Ciphertext>>& cts,
                          const GaloisKeys& galois_keys, const RelinKeys& relin_keys, wire::RequestMsg* request) {
  Status st = SaveRequest(ep, cts, request);
  if (!st.ok()) return st;
  request->galois_keys = SerializeGaloisKeys(ep, galois_keys);
  request->relin_keys = SerializeRelinKeys(ep, relin_keys);
  return OkStatus();
}

namespace detail {
struct CtxDeleter { void operator()(pirb_ctx* c) const { pirb_ctx_destroy(c); } };
struct KeysDeleter { void operator()(pirb_keys* k) const { pirb_keys_destroy(k); } };
inline std::vector<uint64_t> integer_encode(int64_t value, size_t N, uint64_t t) {  // SEAL IntegerEncoder::encode
  std::vector<uint64_t> pt(N, 0);
  const bool neg = value < 0;
  uint64_t v = neg ? (uint64_t)(-value) : (uint64_t)value;
  for (size_t i = 0; v; ++i, v >>= 1)
    if (v & 1) pt[i] = neg ? t - 1 : 1;
  return pt;
}
// page-locked staging that lives as long as the server: the kernels read / write it in place and the captured graph of
// the answer path (keyed on the buffer addresses) is replayed from the second request on
struct PinnedBuf {
  uint64_t* p = nullptr;
  size_t cap = 0;  // limbs
  PinnedBuf() = default;
  PinnedBuf(const PinnedBuf&) = delete;
  PinnedBuf& operator=(const PinnedBuf&) = delete;
  ~PinnedBuf() { if (p) pirb_host_free(p); }
  Status ensure(size_t limbs) {
    if (limbs <= cap) return OkStatus();
    if (p) { pirb_host_free(p); p = nullptr; cap = 0; }
    void* q = nullptr;
    Status st = FromRc(pirb_host_alloc(limbs * sizeof(uint64_t), &q));
    if (!st.ok()) return st;
    p = static_cast<uint64_t*>(q);
    cap = limbs;
    return OkStatus();
  }
};
// 128-bit content fingerprint (four independent multiply-rotate lanes over 64-bit words + the length): identifies a
// client's key material so that its device-resident copy is reused by later requests
struct Fingerprint {
  uint64_t a = 0, b = 0;
  bool operator==(const Fingerprint& o) const { return a == o.a && b == o.b; }
};
inline Fingerprint fingerprint(const void* data, size_t n_bytes, uint64_t salt = 0) {
  const unsigned char* p = static_cast<const unsigned char*>(data);
  uint64_t h[4] = {0x9e3779b97f4a7c15ull ^ salt, 0xbf58476d1ce4e5b9ull, 0x94d049bb133111ebull, 0x2545f4914f6cdd1dull ^ n_bytes};
  auto mix = [](uint64_t h_, uint64_t w) {
    h_ ^= w;
    h_ = (h_ << 27) | (h_ >> 37);
    return h_ * 0xff51afd7ed558ccdull + 0xc4ceb9fe1a85ec53ull;
  };
  size_t i = 0;
  for (; i + 32 <= n_bytes; i += 32) {
    uint64_t w[4];
    std::memcpy(w, p + i, 32);
    h[0] = mix(h[0], w[0]);
    h[1] = mix(h[1], w[1]);
    h[2] = mix(h[2], w[2]);
    h[3] = mix(h[3], w[3]);
  }
  for (int lane = 0; i < n_bytes; i += 8, lane = (lane + 1) & 3) {
    uint64_t w = 0;
    std::memcpy(&w, p + i, std::min<size_t>(8, n_bytes - i));
    h[lane] = mix(h[lane], w);
  }
  Fingerprint f;
  f.a = mix(mix(h[0], h[1]), h[2] ^ 0x1234567);
  f.b = mix(mix(h[3], h[2]), h[0] ^ 0x7654321);
  return f;
}
}  // namespace detail

// ---------------------------------------------------------------------------------------------------------------
// PIRDatabase (database.h:47-127).  One context per GPU: Create(params) / Create(params, device) hold the whole
// database on one device; Create(params, {d0, d1, ...}) shards it by rows of the first dimension across the listed
// devices of this process (SURVEY §8e) — populate() hands every shard the plaintexts it owns.
class PIRDatabase {
 public:
  static StatusOr<std::shared_ptr<PIRDatabase>> Create(std::shared_ptr<PIRParameters> params,
                                                       const std::vector<int>& devices) {
    if (devices.empty()) return InvalidArgumentError("no device given");
    const auto& ep = params->encryption_parameters;
    if (ep.coeff_modulus.size() > PIRB_MAX_MODULI || params->dimensions.size() > PIRB_MAX_DIMS)
      return InvalidArgumentError("too many moduli or dimensions");
    std::shared_ptr<PIRDatabase> db(new PIRDatabase(params));
    for (size_t i = 0; i < devices.size(); ++i) {
      pirb_params p{};
      p.poly_modulus_degree = ep.poly_modulus_degree;
      p.n_moduli = (uint32_t)ep.coeff_modulus.size();
      std::copy(ep.coeff_modulus.begin(), ep.coeff_modulus.end(), p.coeff_modulus);
      p.plain_modulus = ep.plain_modulus;
      p.n_dims = (uint32_t)params->dimensions.size();
      std::copy(params->dimensions.begin(), params->dimensions.end(), p.dims);
      p.num_pt = params->num_pt;
      p.device = devices[i];
      p.shard_index = (uint32_t)i;
      p.shard_count = (uint32_t)devices.size();
      p.use_ciphertext_multiplication = params->use_ciphertext_multiplication ? 1 : 0;
      pirb_ctx* ctx = nullptr;
      Status st = FromRc(pirb_ctx_create(&p, &ctx));
      if (!st.ok()) return st;
      db->ctx_.emplace_back(ctx);
    }
    return db;
  }
  static StatusOr<std::shared_ptr<PIRDatabase>> Create(std::shared_ptr<PIRParameters> params, int device = 0) {
    return Create(std::move(params), std::vector<int>{device});
  }
  template <typename Raw>
  static StatusOr<std::shared_ptr<PIRDatabase>> Create(const std::vector<Raw>& rawdb,
                                                       std::shared_ptr<PIRParameters> params,
                                                       const std::vector<int>& devices = {0}) {
    auto db = Create(params, devices);
    if (!db.ok()) return db.status();
    Status st = (*db)->populate(rawdb);
    if (!st.ok()) return st;
    return db;
  }

  // database.cpp:84-110
  Status populate(const std::vector<std::string>& rawdb) {
    if (rawdb.size() != params_->num_items)
      return InvalidArgumentError("Database size " + std::to_string(rawdb.size()) + " does not match params value " +
                                  std::to_string(params_->num_items));
    const size_t N = params_->encryption_parameters.poly_modulus_degree;
    const size_t ipp = params_->items_per_plaintext;
    StringEncoder encoder(params_->encryption_parameters);
    if (params_->bits_per_coeff > 0) encoder.set_bits_per_coeff(params_->bits_per_coeff);
    const size_t chunk = std::max<size_t>(1, (32u << 20) / (N * 8));
    std::vector<uint64_t> buf, coeffs;
    auto raw_it = rawdb.begin();
    for (size_t start = 0; start < params_->num_pt; start += chunk) {
      const size_t stop = std::min<size_t>(params_->num_pt, start + chunk);
      buf.assign((stop - start) * N, 0);
      for (size_t i = start; i < stop; ++i) {
        auto end_it = (size_t)(rawdb.end() - raw_it) > ipp ? raw_it + ipp : rawdb.end();
        Status st = encoder.encode(raw_it, end_it, coeffs);
        if (!st.ok()) return st;
        std::copy(coeffs.begin(), coeffs.end(), buf.begin() + (i - start) * N);
        raw_it = end_it;
      }
      for (auto& c : ctx_) {  // every shard keeps the plaintexts it owns
        Status st = FromRc(pirb_db_load_coeff(c.get(), buf.data(), start, stop - start));
        if (!st.ok()) return st;
      }
    }
    return OkStatus();
  }
  // database.cpp:60-82
  Status populate(const std::vector<int64_t>& rawdb) {
    if (rawdb.size() != params_->num_items)
      return InvalidArgumentError("Database size " + std::to_string(rawdb.size()) + " does not match params value " +
                                  std::to_string(params_->num_items));
    const size_t N = params_->encryption_parameters.poly_modulus_degree;
    std::vector<uint64_t> buf(rawdb.size() * N);
    for (size_t i = 0; i < rawdb.size(); ++i) {
      auto pt = detail::integer_encode(rawdb[i], N, params_->encryption_parameters.plain_modulus);
      std::copy(pt.begin(), pt.end(), buf.begin() + i * N);
    }
    for (auto& c : ctx_) {
      Status st = FromRc(pirb_db_load_coeff(c.get(), buf.data(), 0, rawdb.size()));
      if (!st.ok()) return st;
    }
    return OkStatus();
  }
  // synthetic NTT-form database (benchmarks): uniform limbs keyed by the global limb index, so the shards of a database
  // are slices of the unsharded fill with the same seed
  Status fill_random(uint64_t seed) {
    for (auto& c : ctx_) {
      Status st = FromRc(pirb_db_fill_random(c.get(), seed));
      if (!st.ok()) return st;
    }
    return OkStatus();
  }

  // database.cpp:290-316 — on the re-encoder path the selection vector is transformed to NTT form in place; in
  // ciphertext-multiplication mode it is left alone and relin_keys (may be null) are applied after every multiplication
  StatusOr<std::vector<Ciphertext>> multiply(std::vector<Ciphertext>& selection_vector,
                                             const RelinKeys* relin_keys = nullptr) const {
    if (ctx_.size() != 1) return InvalidArgumentError("multiply() needs an unsharded database; use PIRServer");
    pirb_ctx* ctx = ctx_[0].get();
    const size_t L = pirb_ct_limbs(ctx);
    std::vector<uint64_t> sv(selection_vector.size() * L);
    for (size_t i = 0; i < selection_vector.size(); ++i) {
      if (selection_vector[i].limbs.size() != L) return InvalidArgumentError("bad ciphertext size");
      std::copy(selection_vector[i].limbs.begin(), selection_vector[i].limbs.end(), sv.begin() + i * L);
    }
    if (params_->use_ciphertext_multiplication) {
      std::unique_ptr<pirb_keys, detail::KeysDeleter> rk;
      if (relin_keys) {
        if (relin_keys->limbs.size() != pirb_key_limbs(ctx)) return InvalidArgumentError("bad relinearization key size");
        pirb_keys* h = nullptr;
        Status st = FromRc(pirb_relin_keys_load(ctx, relin_keys->limbs.data(), &h));
        if (!st.ok()) return st;
        rk.reset(h);
      }
      const size_t polys = pirb_reply_polys(ctx, rk ? 1 : 0), ptL = pirb_pt_limbs(ctx);
      std::vector<Ciphertext> res(1);
      res[0].limbs.assign(polys * ptL, 0);
      uint32_t got = 0;
      Status st = FromRc(pirb_db_multiply_ct(ctx, sv.data(), selection_vector.size(), rk.get(), res[0].limbs.data(),
                                             res[0].limbs.size(), &got));
      if (!st.ok()) return st;
      if (!got) res.clear();
      return res;
    }
    const size_t cap = pirb_reply_cts(ctx);
    std::vector<uint64_t> out(cap * L);
    uint64_t cnt = 0;
    Status st = FromRc(pirb_db_multiply(ctx, sv.data(), selection_vector.size(), out.data(), cap, &cnt));
    if (!st.ok()) return st;
    for (size_t i = 0; i < selection_vector.size(); ++i)
      if (std::memcmp(selection_vector[i].limbs.data(), sv.data() + i * L, L * 8) != 0) {
        std::copy(sv.begin() + i * L, sv.begin() + (i + 1) * L, selection_vector[i].limbs.begin());
        selection_vector[i].is_ntt_form = true;
      }
    std::vector<Ciphertext> res(cnt);
    for (size_t i = 0; i < cnt; ++i) res[i].limbs.assign(out.begin() + i * L, out.begin() + (i + 1) * L);
    return res;
  }

  size_t size() const {  // database.h:94 — plaintexts held, over all shards
    size_t n = 0;
    for (auto& c : ctx_) n += pirb_db_size(c.get());
    return n;
  }

  // database.cpp:318-332 (the parameter-only forms need no device and are what the instance methods use)
  static std::vector<uint32_t> calculate_indices(const PIRParameters& p, uint32_t index) {
    uint32_t pt_index = index / p.items_per_plaintext;
    std::vector<uint32_t> results(p.dimensions.size(), 0);
    for (int i = (int)results.size() - 1; i >= 0; --i) {
      results[i] = pt_index % p.dimensions[i];
      pt_index = pt_index / p.dimensions[i];
    }
    return results;
  }
  static size_t calculate_item_offset(const PIRParameters& p, uint32_t index) {
    const uint32_t pt_index = index / p.items_per_plaintext;
    return (index - (pt_index * p.items_per_plaintext)) * p.bytes_per_item;
  }
  std::vector<uint32_t> calculate_indices(uint32_t index) const { return calculate_indices(*params_, index); }
  size_t calculate_item_offset(uint32_t index) const { return calculate_item_offset(*params_, index); }
  static std::vector<uint32_t> calculate_dimensions(uint32_t db_size, uint32_t num_dimensions) {
    std::vector<uint32_t> r(num_dimensions);
    pirb_calculate_dimensions(db_size, num_dimensions, r.data());
    return r;
  }

  pirb_ctx* handle(size_t shard = 0) const { return ctx_[shard].get(); }
  size_t shard_count() const { return ctx_.size(); }
  const std::shared_ptr<PIRParameters>& params() const { return params_; }

 private:
  explicit PIRDatabase(std::shared_ptr<PIRParameters> p) : params_(std::move(p)) {}
  std::shared_ptr<PIRParameters> params_;
  std::vector<std::unique_ptr<pirb_ctx, detail::CtxDeleter>> ctx_;
};

// ---------------------------------------------------------------------------------------------------------------
// PIRServer (server.h:43-131).  Differences from the reference that a caller can observe are performance only:
//   * a client's Galois keys are uploaded once and found again by a fingerprint of their bytes (the reference
//     deserializes them on every request, server.cpp:46-48);
//   * all queries of a request are answered by one batched device call (the reference loops, server.cpp:60-63);
//   * over a sharded database the queries of a request are spread over the GPUs, every GPU multiplies all of them
//     against its rows, and the exchange runs inside the kernels over NVLink peer memory (pirb_dist_*).
class PIRServer {
 public:
  // server.cpp:35-42.  max_queries_per_gpu: queries one GPU expands per step of the sharded flow.
  static StatusOr<std::unique_ptr<PIRServer>> Create(std::shared_ptr<PIRDatabase> db,
                                                     std::shared_ptr<PIRParameters> params,
                                                     uint32_t max_queries_per_gpu = 8) {
    if (params->num_pt != db->size()) return InvalidArgumentError("database size mismatch");
    std::unique_ptr<PIRServer> s(new PIRServer(std::move(db), std::move(params)));
    const size_t W = s->db_->shard_count();
    if (W > 1) {
      if (s->params_->dimensions.size() < 2)
        return InvalidArgumentError("a sharded PIRServer needs a database of two or more dimensions");
      s->max_local_ = std::max<uint32_t>(1, max_queries_per_gpu);
      std::vector<void*> bases(W, nullptr);
      for (size_t r = 0; r < W; ++r) {
        Status st = FromRc(pirb_dist_create(s->db_->handle(r), s->max_local_, 0, nullptr, &bases[r]));
        if (!st.ok()) return st;
      }
      for (size_t r = 0; r < W; ++r) {
        Status st = FromRc(pirb_dist_attach(s->db_->handle(r), bases.data(), (uint32_t)W, (uint32_t)r));
        if (!st.ok()) return st;
      }
    }
    return s;
  }

  // server.cpp:44-65: all queries of the request in one batched device call
  StatusOr<Response> ProcessRequest(const Request& request) const {
    const detail::Fingerprint fp = KeyFingerprint(request.galois_keys);
    auto keys = FindKeys(fp);
    if (!keys) {
      auto loaded = UploadKeys(request.galois_keys, fp);
      if (!loaded.ok()) return loaded.status();
      keys = *loaded;
    }
    if (params_->use_ciphertext_multiplication)
      return AnswerCt(request.query, *keys, request.relin_keys ? &*request.relin_keys : nullptr);
    return Answer(request.query, *keys);
  }

  // server.cpp:44-65 on the wire: serialized pir.Request in, serialized pir.Response out.  Deserialization failures
  // are InvalidArgument (serialization.h:113-115); relin_keys are parsed for validity and otherwise unused
  // (server.cpp:53-58).  Reply ciphertexts carry the parms_id of the query's first ciphertext.  The serialized key
  // bytes are fingerprinted BEFORE they are parsed: a returning client's keys are neither deserialized nor (for
  // seed-compressed keys) re-expanded.
  StatusOr<std::string> ProcessRequest(const std::string& serialized_request, bool strict_parms_id = false) const {
    wire::RequestView msg;  // views into the caller's bytes: the ~5 MB of key material are not copied
    if (!wire::ParseView(serialized_request, &msg)) return InvalidArgumentError("malformed Request message");
    const EncryptionParameters& ep = params_->encryption_parameters;
    const wire::SealParams sp = ToSealParams(ep);
    auto keys_or = WireKeys(msg);
    if (!keys_or.ok()) return keys_or.status();
    std::shared_ptr<KeySet> keys = *keys_or;
    pirb_ctx* ctx = db_->handle();
    const size_t Q = msg.query.size(), k = ep.coeff_modulus.size() - 1, N = ep.poly_modulus_degree;
    const size_t R = pirb_reply_cts(ctx);
    if (Q == 0) return wire::Serialize(wire::ResponseMsg());
    if (params_->use_ciphertext_multiplication) {
      // server.cpp:53-58, 185-190: here the relinearization keys ARE used; the reply is one ciphertext per query
      Request req;
      wire::parms_id_type pid0 = wire::data_parms_id(sp);
      for (size_t qi = 0; qi < Q; ++qi) {
        req.query.emplace_back();
        for (const auto& blob : msg.query[qi]) {
          wire::parms_id_type pid;
          auto ct = DeserializeCiphertext(ep, std::string(blob), &pid);
          if (!ct.ok()) return ct.status();
          if (strict_parms_id && pid != pid0) return InvalidArgumentError("ciphertext data is invalid");
          if (qi == 0 && req.query[0].empty()) pid0 = pid;
          req.query.back().push_back(std::move(*ct));
        }
      }
      std::optional<RelinKeys> relin;
      if (!msg.relin_keys.empty()) {
        auto rk = DeserializeGaloisKeys(ep, std::string(msg.relin_keys));  // same KSwitchKeys object, one slot
        if (!rk.ok()) return rk.status();
        if (rk->elts.size() != 1) return InvalidArgumentError("relinearization keys must hold exactly one key");
        relin.emplace();
        relin->limbs = std::move(rk->limbs);
      }
      auto resp = AnswerCt(req.query, *keys, relin ? &*relin : nullptr);
      if (!resp.ok()) return resp.status();
      std::string out;
      for (const auto& reply : resp->reply) {
        const size_t polys = reply[0].limbs.size() / (k * N);
        const size_t blob = wire::CiphertextBlobSize(polys, N, k);
        wire::put_tag(out, 1, 2);
        wire::put_varint(out, 1 + wire::varint_size(blob) + blob);
        wire::put_tag(out, 1, 2);
        wire::put_varint(out, blob);
        wire::AppendCiphertextBlob(out, reply[0].limbs.data(), polys, N, k, pid0, false);
      }
      return out;
    }
    const size_t n_ct = msg.query[0].size();
    for (const auto& q : msg.query)
      if (q.size() != n_ct || n_ct != pirb_query_cts(ctx))
        return InvalidArgumentError("Number of ciphertexts doesn't match number of items for oblivious expansion.");
    // ciphertexts are deserialized straight into the page-locked staging buffer and the response is serialized straight
    // out of it: one pass each way, no intermediate Ciphertext objects
    WireReply wr(Q, R, N, k);
    Status st = AnswerSteps(
        Q, n_ct, keys.get(), nullptr,
        [&](size_t qi, uint64_t* dst) { return LoadWireQuery(msg.query[qi], dst, strict_parms_id, &wr); },
        [&](size_t, const uint64_t* src) { AppendWireReply(src, &wr); });
    if (!st.ok()) return st;
    return std::move(wr.out);
  }

  // ProcessRequest for requests of several clients, each with its own Galois keys, in one batched device call
  // (pirb_answer_multi): every Response equals what ProcessRequest returns for that request alone.  The batch fails as a
  // whole if one request is invalid.  On a sharded database and in ciphertext-multiplication mode the requests are
  // answered one by one.
  StatusOr<std::vector<Response>> ProcessRequests(const std::vector<Request>& requests) const {
    std::vector<Response> responses;
    if (db_->shard_count() != 1 || params_->use_ciphertext_multiplication) {
      for (const auto& r : requests) {
        auto resp = ProcessRequest(r);
        if (!resp.ok()) return resp.status();
        responses.push_back(std::move(*resp));
      }
      return responses;
    }
    pirb_ctx* ctx = db_->handle();
    const size_t L = pirb_ct_limbs(ctx), R = pirb_reply_cts(ctx), n_ct = pirb_query_cts(ctx);
    // the batch's key sets stay referenced here until the call returns: the cache may evict them in the meantime
    std::vector<std::shared_ptr<KeySet>> held;
    std::vector<const pirb_keys*> per_query;
    std::vector<std::pair<size_t, size_t>> where;  // batch position -> (request, query of the request)
    for (size_t r = 0; r < requests.size(); ++r) {
      auto keys = KeysFor(requests[r].galois_keys);
      if (!keys.ok()) return keys.status();
      held.push_back(*keys);
      const auto& query = requests[r].query;
      for (size_t i = 0; i < query.size(); ++i) {
        if (query[i].size() != n_ct)
          return InvalidArgumentError("Number of ciphertexts doesn't match number of items for oblivious expansion.");
        for (size_t c = 0; c < n_ct; ++c)
          if (query[i][c].limbs.size() != L) return InvalidArgumentError("bad ciphertext size");
        per_query.push_back(held.back()->per_shard[0].get());
        where.emplace_back(r, i);
      }
    }
    responses.resize(requests.size());
    if (per_query.empty()) return responses;
    for (size_t r = 0; r < requests.size(); ++r) responses[r].reply.resize(requests[r].query.size());
    Status st = AnswerSteps(
        per_query.size(), n_ct, nullptr, per_query.data(),
        [&](size_t qi, uint64_t* dst) -> Status {
          const auto& q = requests[where[qi].first].query[where[qi].second];
          for (size_t c = 0; c < n_ct; ++c) std::memcpy(dst + c * L, q[c].limbs.data(), L * sizeof(uint64_t));
          return OkStatus();
        },
        [&](size_t qi, const uint64_t* src) {
          auto& reply = responses[where[qi].first].reply[where[qi].second];
          reply.resize(R);
          for (size_t c = 0; c < R; ++c) reply[c].limbs.assign(src + c * L, src + (c + 1) * L);
        });
    if (!st.ok()) return st;
    return responses;
  }

  // The wire form of ProcessRequests: serialized pir.Requests in, serialized pir.Responses out, each byte-identical to
  // what ProcessRequest(serialized, strict_parms_id) returns for it alone.
  StatusOr<std::vector<std::string>> ProcessRequests(const std::vector<std::string>& serialized,
                                                      bool strict_parms_id = false) const {
    std::vector<std::string> outs;
    if (db_->shard_count() != 1 || params_->use_ciphertext_multiplication) {
      for (const auto& s : serialized) {
        auto out = ProcessRequest(s, strict_parms_id);
        if (!out.ok()) return out.status();
        outs.push_back(std::move(*out));
      }
      return outs;
    }
    const EncryptionParameters& ep = params_->encryption_parameters;
    pirb_ctx* ctx = db_->handle();
    const size_t k = ep.coeff_modulus.size() - 1, N = ep.poly_modulus_degree, R = pirb_reply_cts(ctx);
    const size_t n_ct = pirb_query_cts(ctx);
    std::vector<wire::RequestView> msgs(serialized.size());
    std::vector<std::shared_ptr<KeySet>> held;  // see ProcessRequests(const std::vector<Request>&)
    std::vector<WireReply> replies;
    std::vector<const pirb_keys*> per_query;
    std::vector<std::pair<size_t, size_t>> where;
    for (size_t r = 0; r < serialized.size(); ++r) {
      if (!wire::ParseView(serialized[r], &msgs[r])) return InvalidArgumentError("malformed Request message");
      auto keys = WireKeys(msgs[r]);
      if (!keys.ok()) return keys.status();
      held.push_back(*keys);
      const size_t Q = msgs[r].query.size();
      for (size_t i = 0; i < Q; ++i) {
        if (msgs[r].query[i].size() != n_ct)
          return InvalidArgumentError("Number of ciphertexts doesn't match number of items for oblivious expansion.");
        per_query.push_back(held.back()->per_shard[0].get());
        where.emplace_back(r, i);
      }
      replies.emplace_back(Q, R, N, k);
    }
    Status st = per_query.empty() ? OkStatus() : AnswerSteps(
        per_query.size(), n_ct, nullptr, per_query.data(),
        [&](size_t qi, uint64_t* dst) {
          const auto [r, i] = where[qi];
          return LoadWireQuery(msgs[r].query[i], dst, strict_parms_id, &replies[r]);
        },
        [&](size_t qi, const uint64_t* src) { AppendWireReply(src, &replies[where[qi].first]); });
    if (!st.ok()) return st;
    for (size_t r = 0; r < serialized.size(); ++r)
      outs.push_back(msgs[r].query.empty() ? wire::Serialize(wire::ResponseMsg()) : std::move(replies[r].out));
    return outs;
  }

  // server.cpp:67-76
  Status substitute_power_x_inplace(Ciphertext& ct, uint32_t power, const GaloisKeys& gal_keys) const {
    auto keys = KeysFor(gal_keys);
    if (!keys.ok()) return keys.status();
    return FromRc(pirb_substitute(db_->handle(), (*keys)->per_shard[0].get(), ct.data(), power));
  }
  // server.cpp:78-103
  void multiply_inverse_power_of_x(const Ciphertext& encrypted, uint32_t k, Ciphertext& destination) const {
    destination = encrypted;
    pirb_mul_inv_pow_x(db_->handle(), encrypted.data(), k, destination.data());
  }
  // server.cpp:105-146
  StatusOr<std::vector<Ciphertext>> oblivious_expansion(const Ciphertext& ct, size_t num_items,
                                                        const GaloisKeys& gal_keys) const {
    return Expand(ct.limbs.data(), 1, num_items, 1, gal_keys);
  }
  // server.cpp:148-171
  StatusOr<std::vector<Ciphertext>> oblivious_expansion(const std::vector<Ciphertext>& cts, size_t total_items,
                                                        const GaloisKeys& gal_keys) const {
    const size_t L = pirb_ct_limbs(db_->handle());
    std::vector<uint64_t> in(cts.size() * L);
    for (size_t i = 0; i < cts.size(); ++i) std::copy(cts[i].limbs.begin(), cts[i].limbs.end(), in.begin() + i * L);
    return Expand(in.data(), cts.size(), total_items, 0, gal_keys);
  }

  void set_key_cache_capacity(size_t n) { key_cache_capacity_ = std::max<size_t>(1, n); }
  size_t key_cache_hits() const { return key_hits_; }

 private:
  struct KeySet {  // one client's Galois keys, resident on every shard's device
    std::vector<std::unique_ptr<pirb_keys, detail::KeysDeleter>> per_shard;
  };
  PIRServer(std::shared_ptr<PIRDatabase> db, std::shared_ptr<PIRParameters> params)
      : db_(std::move(db)), params_(std::move(params)) {}

  static detail::Fingerprint KeyFingerprint(const GaloisKeys& gk) {
    detail::Fingerprint a = detail::fingerprint(gk.limbs.data(), gk.limbs.size() * sizeof(uint64_t));
    detail::Fingerprint b = detail::fingerprint(gk.elts.data(), gk.elts.size() * sizeof(uint32_t), a.a);
    return detail::Fingerprint{a.a ^ b.b, a.b ^ b.a};
  }
  std::shared_ptr<KeySet> FindKeys(const detail::Fingerprint& fp) const {
    for (auto it = key_cache_.begin(); it != key_cache_.end(); ++it)
      if (it->first == fp) {
        auto hit = *it;
        key_cache_.erase(it);
        key_cache_.insert(key_cache_.begin(), hit);  // most recently used first
        ++key_hits_;
        return hit.second;
      }
    return nullptr;
  }
  StatusOr<std::shared_ptr<KeySet>> UploadKeys(const GaloisKeys& gk, const detail::Fingerprint& fp) const {
    if (gk.limbs.size() != gk.elts.size() * pirb_key_limbs(db_->handle()))
      return InvalidArgumentError("Galois key data has the wrong size");
    auto ks = std::make_shared<KeySet>();
    for (size_t r = 0; r < db_->shard_count(); ++r) {
      pirb_keys* k = nullptr;
      Status st = FromRc(pirb_keys_load(db_->handle(r), gk.elts.data(), (uint32_t)gk.elts.size(), gk.limbs.data(), &k));
      ks->per_shard.emplace_back(k);
      if (!st.ok()) return st;
    }
    key_cache_.insert(key_cache_.begin(), std::make_pair(fp, ks));
    while (key_cache_.size() > key_cache_capacity_) key_cache_.pop_back();
    return ks;
  }
  StatusOr<std::shared_ptr<KeySet>> KeysFor(const GaloisKeys& gk) const {
    const detail::Fingerprint fp = KeyFingerprint(gk);
    if (auto hit = FindKeys(fp)) return hit;
    return UploadKeys(gk, fp);
  }

  // processQuery for every query of a request (server.cpp:60-63, 173-195)
  StatusOr<Response> Answer(const std::vector<std::vector<Ciphertext>>& query, const KeySet& keys) const {
    pirb_ctx* ctx = db_->handle();
    Response response;
    if (query.empty()) return response;
    const size_t L = pirb_ct_limbs(ctx), n_ct = query[0].size(), R = pirb_reply_cts(ctx), Q = query.size();
    for (size_t i = 0; i < Q; ++i) {
      if (query[i].size() != n_ct || n_ct != pirb_query_cts(ctx))
        return InvalidArgumentError("Number of ciphertexts doesn't match number of items for oblivious expansion.");
      for (size_t c = 0; c < n_ct; ++c)
        if (query[i][c].limbs.size() != L) return InvalidArgumentError("bad ciphertext size");
    }
    response.reply.resize(Q);
    Status st = AnswerSteps(
        Q, n_ct, &keys, nullptr,
        [&](size_t qi, uint64_t* dst) -> Status {
          for (size_t c = 0; c < n_ct; ++c) std::memcpy(dst + c * L, query[qi][c].limbs.data(), L * sizeof(uint64_t));
          return OkStatus();
        },
        [&](size_t qi, const uint64_t* src) {
          response.reply[qi].resize(R);
          for (size_t c = 0; c < R; ++c) response.reply[qi][c].limbs.assign(src + c * L, src + (c + 1) * L);
        });
    if (!st.ok()) return st;
    return response;
  }
  // processQuery in ciphertext-multiplication mode (server.cpp:173-195 with database.cpp:202-211): one reply ciphertext
  // per query, of 2 polynomials when relinearization keys are given, else one more per upper dimension
  StatusOr<Response> AnswerCt(const std::vector<std::vector<Ciphertext>>& query, const KeySet& keys,
                              const RelinKeys* relin) const {
    if (db_->shard_count() != 1) return InvalidArgumentError("ciphertext-multiplication mode runs on one GPU");
    pirb_ctx* ctx = db_->handle();
    Response response;
    if (query.empty()) return response;
    const size_t L = pirb_ct_limbs(ctx), ptL = pirb_pt_limbs(ctx), n_ct = query[0].size(), Q = query.size();
    std::vector<uint64_t> q(Q * n_ct * L);
    for (size_t i = 0; i < Q; ++i) {
      if (query[i].size() != n_ct || n_ct != pirb_query_cts(ctx))
        return InvalidArgumentError("Number of ciphertexts doesn't match number of items for oblivious expansion.");
      for (size_t c = 0; c < n_ct; ++c) {
        if (query[i][c].limbs.size() != L) return InvalidArgumentError("bad ciphertext size");
        std::memcpy(q.data() + (i * n_ct + c) * L, query[i][c].limbs.data(), L * sizeof(uint64_t));
      }
    }
    std::unique_ptr<pirb_keys, detail::KeysDeleter> rk;
    if (relin) {
      if (relin->limbs.size() != pirb_key_limbs(ctx)) return InvalidArgumentError("bad relinearization key size");
      pirb_keys* h = nullptr;
      Status st = FromRc(pirb_relin_keys_load(ctx, relin->limbs.data(), &h));
      if (!st.ok()) return st;
      rk.reset(h);
    }
    const size_t polys = pirb_reply_polys(ctx, rk ? 1 : 0);
    std::vector<uint64_t> r(Q * polys * ptL);
    Status st = FromRc(pirb_answer_ct(ctx, keys.per_shard[0].get(), rk.get(), q.data(), (uint32_t)Q, n_ct, r.data()));
    if (!st.ok()) return st;
    response.reply.resize(Q);
    for (size_t i = 0; i < Q; ++i) {
      response.reply[i].resize(1);
      response.reply[i][0].limbs.assign(r.begin() + i * polys * ptL, r.begin() + (i + 1) * polys * ptL);
    }
    return response;
  }
  // The step engine behind both forms of ProcessRequest and ProcessRequests: fill(qi, dst) writes query qi's n_ct
  // ciphertexts into the page-locked staging buffer, drain(qi, src) consumes its reply ciphertexts from there, in query
  // order.  Either one key set for every query, or (unsharded only) one Galois-key handle per query in per_query.
  template <typename Fill, typename Drain>
  Status AnswerSteps(size_t Q, size_t n_ct, const KeySet* keys, const pirb_keys* const* per_query, Fill&& fill,
                     Drain&& drain) const {
    pirb_ctx* ctx = db_->handle();
    const size_t L = pirb_ct_limbs(ctx), R = pirb_reply_cts(ctx);
    const size_t W = db_->shard_count();
    // sharded: every GPU takes the same number of queries per step (the last step is padded with zero queries)
    const size_t ql = W > 1 ? std::min<size_t>(max_local_, (Q + W - 1) / W) : Q;
    const size_t per_step = W > 1 ? W * ql : Q;
    const size_t n_steps = (Q + per_step - 1) / per_step;
    Status st = q_pin_.ensure(per_step * n_ct * L);
    if (!st.ok()) return st;
    st = r_pin_.ensure(per_step * R * L);
    if (!st.ok()) return st;
    for (size_t step = 0; step < n_steps; ++step) {
      const size_t q0 = step * per_step, qn = std::min(per_step, Q - q0);
      for (size_t i = 0; i < per_step; ++i) {
        uint64_t* dst = q_pin_.p + i * n_ct * L;
        if (i < qn) {
          st = fill(q0 + i, dst);
          if (!st.ok()) return st;
        } else {
          std::memset(dst, 0, n_ct * L * sizeof(uint64_t));
        }
      }
      if (W == 1) {
        st = FromRc(per_query ? pirb_answer_multi(ctx, per_query + q0, q_pin_.p, (uint32_t)qn, n_ct, r_pin_.p)
                              : pirb_answer(ctx, keys->per_shard[0].get(), q_pin_.p, (uint32_t)qn, n_ct, r_pin_.p));
        if (!st.ok()) return st;
      } else {
        // one host thread drives all ranks: nothing that may synchronise a device (allocations, first launches) may
        // happen between one rank's launches and the next's, so every rank is prepared before the first step
        for (size_t r = 0; r < W; ++r) {
          st = FromRc(pirb_dist_prepare(db_->handle(r), keys->per_shard[r].get(), (uint32_t)ql));
          if (!st.ok()) return st;
        }
        for (size_t r = 0; r < W; ++r) {
          st = FromRc(pirb_dist_answer_dev(db_->handle(r), keys->per_shard[r].get(), q_pin_.p + r * ql * n_ct * L,
                                           (uint32_t)ql, n_ct, r_pin_.p + r * ql * R * L, nullptr));
          if (!st.ok()) return st;
        }
        for (size_t r = 0; r < W; ++r) {
          st = FromRc(pirb_sync(db_->handle(r)));
          if (!st.ok()) return st;
        }
        for (size_t r = 0; r < W; ++r) {
          st = FromRc(pirb_dist_status(db_->handle(r)));
          if (!st.ok()) return st;
        }
      }
      for (size_t i = 0; i < qn; ++i) drain(q0 + i, r_pin_.p + i * R * L);
    }
    return OkStatus();
  }
  // The key set of a wire request: found by a fingerprint of the serialized keys, else deserialized and uploaded; its
  // relinearization keys, if any, are parsed for validity only (server.cpp:53-58), once per distinct key blob.
  StatusOr<std::shared_ptr<KeySet>> WireKeys(const wire::RequestView& msg) const {
    const EncryptionParameters& ep = params_->encryption_parameters;
    const detail::Fingerprint fp = detail::fingerprint(msg.galois_keys.data(), msg.galois_keys.size(), /*salt=*/1);
    auto keys = FindKeys(fp);
    if (!keys) {
      auto gk = DeserializeGaloisKeys(ep, std::string(msg.galois_keys));
      if (!gk.ok()) return gk.status();
      auto loaded = UploadKeys(*gk, fp);
      if (!loaded.ok()) return loaded.status();
      keys = *loaded;
    }
    if (!msg.relin_keys.empty()) {
      const detail::Fingerprint rfp = detail::fingerprint(msg.relin_keys.data(), msg.relin_keys.size(), /*salt=*/2);
      if (!(rfp == last_relin_ok_)) {
        std::string err;
        wire::KSwitchKeysData rk;
        if (!wire::LoadKSwitchKeys(std::string(msg.relin_keys), ToSealParams(ep), &rk, &err, /*keep_data=*/false))
          return InvalidArgumentError(err);
        last_relin_ok_ = rfp;
      }
    }
    return keys;
  }
  // One serialized Response under construction: its replies carry the parms_id of the request's first ciphertext.
  struct WireReply {
    size_t R, N, k, blob, inner;
    wire::parms_id_type pid = {};
    bool first = true;
    std::string out;
    WireReply(size_t Q, size_t R_, size_t N_, size_t k_)
        : R(R_), N(N_), k(k_), blob(wire::CiphertextBlobSize(2, N_, k_)), inner(R_ * (1 + wire::varint_size(blob) + blob)) {
      out.reserve(Q * (1 + wire::varint_size(inner) + inner));
    }
  };
  // Deserializes one query's ciphertexts of a wire request into dst
  Status LoadWireQuery(const std::vector<std::string_view>& cts, uint64_t* dst, bool strict_parms_id, WireReply* wr) const {
    const EncryptionParameters& ep = params_->encryption_parameters;
    const size_t L = pirb_ct_limbs(db_->handle());
    const wire::parms_id_type data_pid = wire::data_parms_id(ToSealParams(ep));
    if (wr->first) wr->pid = data_pid;
    std::string err;
    for (size_t c = 0; c < cts.size(); ++c) {
      wire::CiphertextData meta;
      if (!wire::LoadCiphertextTo(cts[c], (uint32_t)wr->N, ep.coeff_modulus.data(), wr->k, dst + c * L, &meta, &err))
        return InvalidArgumentError(err);
      if (strict_parms_id && meta.parms_id != data_pid) return InvalidArgumentError("ciphertext data is invalid");
      if (wr->first) { wr->pid = meta.parms_id; wr->first = false; }
    }
    return OkStatus();
  }
  // Appends one query's reply ciphertexts (at src) to the serialized Response
  void AppendWireReply(const uint64_t* src, WireReply* wr) const {
    const size_t L = pirb_ct_limbs(db_->handle());
    wire::put_tag(wr->out, 1, 2);
    wire::put_varint(wr->out, wr->inner);
    for (size_t c = 0; c < wr->R; ++c) {
      wire::put_tag(wr->out, 1, 2);
      wire::put_varint(wr->out, wr->blob);
      wire::AppendCiphertextBlob(wr->out, src + c * L, 2, wr->N, wr->k, wr->pid, false);
    }
  }
  StatusOr<std::vector<Ciphertext>> Expand(const uint64_t* cts, size_t n_ct, size_t total, int single,
                                           const GaloisKeys& gal_keys) const {
    auto keys = KeysFor(gal_keys);
    if (!keys.ok()) return keys.status();
    const size_t L = pirb_ct_limbs(db_->handle());
    std::vector<uint64_t> out(std::max<size_t>(1, total) * L);
    Status st = FromRc(pirb_expand(db_->handle(), (*keys)->per_shard[0].get(), cts, n_ct, total, single, out.data()));
    if (!st.ok()) return st;
    std::vector<Ciphertext> res(total);
    for (size_t i = 0; i < total; ++i) res[i].limbs.assign(out.begin() + i * L, out.begin() + (i + 1) * L);
    return res;
  }
  std::shared_ptr<PIRDatabase> db_;
  std::shared_ptr<PIRParameters> params_;
  uint32_t max_local_ = 8;
  // ProcessRequest is const like the reference's, but reuses staging and cached keys: one host thread at a time
  mutable detail::PinnedBuf q_pin_, r_pin_;
  mutable std::vector<std::pair<detail::Fingerprint, std::shared_ptr<KeySet>>> key_cache_;
  mutable size_t key_cache_capacity_ = 4, key_hits_ = 0;
  mutable detail::Fingerprint last_relin_ok_;
};

}  // namespace pir
