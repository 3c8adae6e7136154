// PIRServer::ProcessRequests (pir_b200/cpp/pir_b200.hpp): requests of several clients, each with its own Galois keys,
// answered in one batched call.  Both overloads must return, byte for byte, what ProcessRequest returns for each request
// alone (the wire form included), and the oracle's answer with that client's keys; a key cache smaller than the batch
// must not free keys the batch uses; a ciphertext-multiplication server answers request by request.
#include <cstdio>
#include <cstdlib>
#include <random>

#include "../../oracle/pir_oracle.hpp"
#include "../../pir_b200/cpp/pir_b200.hpp"

#define CHECK(cond, msg)                                            \
  do {                                                              \
    if (!(cond)) {                                                  \
      std::fprintf(stderr, "FAIL %s:%d %s\n", __FILE__, __LINE__, msg); \
      return 1;                                                     \
    }                                                               \
  } while (0)

namespace {

struct Client {
  orc::SecretKey sk;
  orc::PublicKey pk;
  pir::GaloisKeys gk;
};

Client make_client(const orc::Context& octx, const pir::EncryptionParameters& ep, uint64_t seed) {
  orc::Rng r(seed);
  Client c;
  c.sk = orc::gen_secret_key(octx, r);
  c.pk = orc::gen_public_key(octx, c.sk, r);
  c.gk.elts = pir::generate_galois_elts(ep.poly_modulus_degree);
  const size_t key_limbs = octx.k * 2 * (octx.k + 1) * octx.N;
  c.gk.limbs.resize(c.gk.elts.size() * key_limbs);
  for (size_t i = 0; i < c.gk.elts.size(); ++i)
    orc::gen_galois_key(octx, c.sk, c.gk.elts[i], r, c.gk.limbs.data() + i * key_limbs);
  return c;
}

// PIRClient::createQueryFor (client.cpp:92-144) for dim_sum <= N
pir::Ciphertext make_query(const orc::Context& octx, orc::Crypto& crypto, const Client& cl, const pir::PIRDatabase& db,
                           const pir::PIRParameters& p, uint32_t index, orc::Rng& r) {
  const size_t N = octx.N;
  auto indices = db.calculate_indices(index);
  size_t dim_sum = 0;
  for (auto v : p.dimensions) dim_sum += v;
  const uint64_t m_inv = orc::invmod(pirb_next_power_two(dim_sum) % p.encryption_parameters.plain_modulus,
                                     orc::Modulus(p.encryption_parameters.plain_modulus));
  std::vector<uint64_t> pt(N, 0);
  size_t offset = 0;
  for (size_t i = 0; i < indices.size(); ++i) {
    pt[offset + indices[i]] = m_inv;
    offset += p.dimensions[i];
  }
  pir::Ciphertext ct;
  ct.limbs.resize(octx.ct_limbs());
  crypto.encrypt(cl.pk, pt.data(), N, r, ct.data());
  return ct;
}

bool same_response(const pir::Response& a, const pir::Response& b) {
  if (a.reply.size() != b.reply.size()) return false;
  for (size_t i = 0; i < a.reply.size(); ++i) {
    if (a.reply[i].size() != b.reply[i].size()) return false;
    for (size_t c = 0; c < a.reply[i].size(); ++c)
      if (a.reply[i][c].limbs != b.reply[i][c].limbs) return false;
  }
  return true;
}

struct Setup {
  pir::EncryptionParameters ep;
  std::shared_ptr<pir::PIRParameters> params;
  std::vector<std::string> items;
  std::shared_ptr<pir::PIRDatabase> db;
};

int make_setup(Setup* s, size_t dbsize, size_t d, bool ct_mode) {
  s->ep = pir::GenerateEncryptionParams(4096, 20);
  auto params_or = pir::CreatePIRParameters(dbsize, 64, d, s->ep, ct_mode);
  CHECK(params_or.ok(), "CreatePIRParameters");
  s->params = *params_or;
  std::mt19937_64 rng(dbsize * 7 + d);
  s->items.assign(dbsize, std::string(s->params->bytes_per_item, 0));
  for (auto& it : s->items)
    for (auto& ch : it) ch = (char)(rng() & 0xff);
  auto db_or = pir::PIRDatabase::Create(s->items, s->params);
  CHECK(db_or.ok(), db_or.status().message().c_str());
  s->db = *db_or;
  return 0;
}

// requests: order[i] = client of request i, sizes[i] = its queries
std::vector<pir::Request> make_requests(const orc::Context& octx, orc::Crypto& crypto, const std::vector<Client>& cls,
                                        const Setup& s, const std::vector<int>& order, const std::vector<int>& sizes,
                                        std::vector<std::vector<uint32_t>>* idx, uint64_t seed) {
  orc::Rng r(seed);
  std::mt19937_64 pick(seed);
  std::vector<pir::Request> reqs;
  idx->clear();
  for (size_t i = 0; i < order.size(); ++i) {
    pir::Request q;
    q.galois_keys = cls[order[i]].gk;
    idx->emplace_back();
    for (int j = 0; j < sizes[i]; ++j) {
      const uint32_t index = (uint32_t)(pick() % s.params->num_items);
      idx->back().push_back(index);
      q.query.push_back({make_query(octx, crypto, cls[order[i]], *s.db, *s.params, index, r)});
    }
    reqs.push_back(std::move(q));
  }
  return reqs;
}

// ProcessRequests(requests) against ProcessRequest(request) and (check_oracle) the oracle with that client's keys
int check_batch(const pir::PIRServer& server, const std::vector<pir::Request>& reqs, const orc::Context& octx,
                const std::vector<uint64_t>& db_ntt, const Setup& s, bool check_oracle, const char* tag) {
  auto batch = server.ProcessRequests(reqs);
  CHECK(batch.ok(), batch.status().message().c_str());
  CHECK(batch->size() == reqs.size(), "one response per request");
  for (size_t r = 0; r < reqs.size(); ++r) {
    auto alone = server.ProcessRequest(reqs[r]);
    CHECK(alone.ok(), alone.status().message().c_str());
    CHECK(same_response((*batch)[r], *alone), tag);
    if (!check_oracle) continue;
    orc::GaloisKeys ogk;
    ogk.elts = reqs[r].galois_keys.elts;
    ogk.data = reqs[r].galois_keys.limbs;
    for (size_t i = 0; i < reqs[r].query.size(); ++i) {
      std::vector<uint64_t> want;
      CHECK(orc::process_query(octx, db_ntt.data(), s.params->num_pt, s.params->dimensions.data(),
                               s.params->dimensions.size(), ogk, reqs[r].query[i][0].data(), 1, want) == 0,
            "oracle process_query");
      const auto& got = (*batch)[r].reply[i];
      CHECK(want.size() == got.size() * octx.ct_limbs(), "reply count");
      for (size_t c = 0; c < got.size(); ++c)
        CHECK(std::memcmp(got[c].data(), want.data() + c * octx.ct_limbs(), octx.ct_limbs() * 8) == 0,
              "batched reply differs from the oracle");
    }
  }
  return 0;
}

}  // namespace

int main() {
  Setup s;
  if (make_setup(&s, 60, 2, false)) return 1;
  orc::Context octx(s.ep.poly_modulus_degree, s.ep.coeff_modulus, s.ep.plain_modulus);
  orc::Crypto crypto(octx);
  std::vector<uint64_t> db_ntt(s.params->num_pt * octx.pt_limbs()), coeffs;
  pir::StringEncoder enc(s.ep);
  for (size_t i = 0; i < s.params->num_pt; ++i) {
    auto b = s.items.begin() + i * s.params->items_per_plaintext;
    auto e = (size_t)(s.items.end() - b) > s.params->items_per_plaintext ? b + s.params->items_per_plaintext : s.items.end();
    CHECK(enc.encode(b, e, coeffs).ok(), "encode");
    orc::plain_to_ntt(octx, coeffs.data(), coeffs.size(), db_ntt.data() + i * octx.pt_limbs());
  }
  std::vector<Client> cls;
  for (int i = 0; i < 5; ++i) cls.push_back(make_client(octx, s.ep, 900 + i));
  std::vector<std::vector<uint32_t>> idx;

  // ---- structured requests: clients A, B, A, C, D, E, B (adjacent queries of different clients) ----
  {
    auto server_or = pir::PIRServer::Create(s.db, s.params);
    CHECK(server_or.ok(), server_or.status().message().c_str());
    auto reqs = make_requests(octx, crypto, cls, s, {0, 1, 0, 2, 3, 4, 1}, {1, 2, 1, 2, 1, 1, 1}, &idx, 1);
    if (check_batch(**server_or, reqs, octx, db_ntt, s, true, "ProcessRequests differs from ProcessRequest")) return 1;
    std::printf("ok: ProcessRequests, 7 requests of 5 clients (9 queries): per-request and oracle parity\n");

    // ---- the wire form: byte-identical to the single-request wire path ----
    std::vector<std::string> wire_reqs;
    for (const auto& r : reqs) {
      pir::wire::RequestMsg msg;
      msg.galois_keys = pir::SerializeGaloisKeys(s.ep, r.galois_keys);
      for (const auto& q : r.query) {
        msg.query.emplace_back();
        msg.query.back().ct.push_back(pir::SerializeCiphertext(s.ep, q[0]));
      }
      wire_reqs.push_back(pir::wire::Serialize(msg));
    }
    wire_reqs.push_back(pir::wire::Serialize([&] {  // a request without queries, keys of client A
      pir::wire::RequestMsg m;
      m.galois_keys = pir::SerializeGaloisKeys(s.ep, cls[0].gk);
      return m;
    }()));
    for (bool strict : {false, true}) {
      auto batch = (*server_or)->ProcessRequests(wire_reqs, strict);
      CHECK(batch.ok(), batch.status().message().c_str());
      CHECK(batch->size() == wire_reqs.size(), "one wire response per request");
      for (size_t r = 0; r < wire_reqs.size(); ++r) {
        auto alone = (*server_or)->ProcessRequest(wire_reqs[r], strict);
        CHECK(alone.ok(), alone.status().message().c_str());
        CHECK((*batch)[r] == *alone, "wire ProcessRequests differs from the wire ProcessRequest");
      }
    }
    // the wire replies decode to the structured ones
    auto batch = (*server_or)->ProcessRequests(wire_reqs);
    for (size_t r = 0; r < reqs.size(); ++r) {
      pir::wire::ResponseMsg rmsg;
      CHECK(pir::wire::Parse((*batch)[r], &rmsg) && rmsg.reply.size() == reqs[r].query.size(), "Response parse");
      auto alone = (*server_or)->ProcessRequest(reqs[r]);
      for (size_t i = 0; i < rmsg.reply.size(); ++i)
        for (size_t c = 0; c < rmsg.reply[i].ct.size(); ++c) {
          auto ct = pir::DeserializeCiphertext(s.ep, rmsg.reply[i].ct[c]);
          CHECK(ct.ok() && ct->limbs == alone->reply[i][c].limbs, "wire reply differs from the structured reply");
        }
    }
    // a malformed request fails the batch with InvalidArgument
    auto bad = (*server_or)->ProcessRequests({wire_reqs[0], wire_reqs[1].substr(0, wire_reqs[1].size() / 2)});
    CHECK(!bad.ok() && bad.status().code() == PIRB_INVALID_ARGUMENT, "truncated request in a batch");
    std::printf("ok: wire ProcessRequests byte-identical to ProcessRequest(serialized), strict and not\n");
  }

  // ---- a key cache of 2 with 5 clients in one call ----
  {
    auto server_or = pir::PIRServer::Create(s.db, s.params);
    CHECK(server_or.ok(), server_or.status().message().c_str());
    (*server_or)->set_key_cache_capacity(2);
    auto reqs = make_requests(octx, crypto, cls, s, {0, 1, 2, 3, 4, 0}, {1, 1, 1, 1, 1, 1}, &idx, 2);
    if (check_batch(**server_or, reqs, octx, db_ntt, s, true, "cache of 2: ProcessRequests differs")) return 1;
    std::printf("ok: key cache of 2, 5 clients in one call\n");
  }

  // ---- ciphertext-multiplication mode: answered request by request ----
  {
    Setup c;
    if (make_setup(&c, 30, 2, true)) return 1;
    auto server_or = pir::PIRServer::Create(c.db, c.params);
    CHECK(server_or.ok(), server_or.status().message().c_str());
    auto reqs = make_requests(octx, crypto, cls, c, {0, 1, 0}, {1, 2, 1}, &idx, 3);
    if (check_batch(**server_or, reqs, octx, db_ntt, c, false, "CT mode: ProcessRequests differs")) return 1;
    std::printf("ok: ciphertext-multiplication server answers ProcessRequests request by request\n");
  }
  std::printf("ALL OK\n");
  return 0;
}
