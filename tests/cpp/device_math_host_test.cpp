// CPU-only test of the DEVICE arithmetic: pir_b200/csrc/pirb_device.cuh is compiled for the host (the intrinsics it
// uses are IEEE-754 operations with exact host equivalents) and its exactness claims (DESIGN.md §4.1) are checked
// against 128-bit integer arithmetic and the oracle's transforms:
//   * f64_modmul with a table companion (w/q) and with the on-the-fly companion w * (1/q): result integer-valued,
//     congruent to y*w, |t| <= 0.54 q / 0.57 q, on random AND adversarial inputs (quotients next to half-integers,
//     |y| at the 2^48 limit, w = q-1);
//   * f64_canon, the u64 <-> double conversions, the FP64 and 24-bit Karatsuba multiply-accumulate chains at their
//     maximum length, Barrett / Shoup reductions;
//   * the shared-memory NTT passes (swizzle, radix-8 schedule, twiddles from the pair table and from the w-only table the
//     cluster kernel stages in shared memory), emulated thread by thread and pass by pass, against the oracle's forward /
//     inverse negacyclic NTT;  the Galois gather against the oracle's apply_galois.
// Nothing here replaces the GPU parity tests: it pins the math of the kernels where no GPU is available.
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <random>
#include <vector>

#include <cuda_runtime.h>

// host stand-ins for the device intrinsics used by the arithmetic helpers (all exact IEEE-754 / integer operations)
static inline unsigned long long __umul64hi(unsigned long long a, unsigned long long b) {
  return (unsigned long long)(((unsigned __int128)a * b) >> 64);
}
static inline double __dmul_rn(double a, double b) { return a * b; }
static inline double __dadd_rn(double a, double b) { return a + b; }
static inline double __fma_rn(double a, double b, double c) { return std::fma(a, b, c); }
static inline double __longlong_as_double(long long v) { double d; std::memcpy(&d, &v, 8); return d; }
static inline long long __double_as_longlong(double d) { long long v; std::memcpy(&v, &d, 8); return v; }
static inline double __hiloint2double(int hi, int lo) {
  const unsigned long long v = ((unsigned long long)(unsigned)hi << 32) | (unsigned)lo;
  double d;
  std::memcpy(&d, &v, 8);
  return d;
}
template <typename T>
static inline T __ldg(const T* p) { return *p; }
static inline void __syncthreads() {}
static inline size_t __cvta_generic_to_shared(const void* p) { return (size_t)p; }

#include "../../oracle/pir_oracle.hpp"
#include "../../pir_b200/csrc/host_math.h"
#include "../../pir_b200/csrc/pirb_device.cuh"
#include "../../pir_b200/csrc/tc_plan.h"

typedef unsigned __int128 u128;
typedef __int128 i128;

#define CHECK(cond, ...)                                       \
  do {                                                         \
    if (!(cond)) {                                             \
      std::fprintf(stderr, "FAIL %s:%d ", __FILE__, __LINE__); \
      std::fprintf(stderr, __VA_ARGS__);                       \
      std::fprintf(stderr, "\n");                              \
      return 1;                                                \
    }                                                          \
  } while (0)

static bool is_integer(double v) { return std::nearbyint(v) == v; }
static u64 mod_i128(i128 v, u64 q) {
  i128 r = v % (i128)q;
  if (r < 0) r += q;
  return (u64)r;
}

static int check_modmul(u64 q, std::mt19937_64& rng, double* worst_table, double* worst_fly) {
  const double qd = (double)q, qinv = 1.0 / qd;
  auto one = [&](double y, u64 w) -> int {
    const double wd = (double)w;
    for (int fly = 0; fly < 2; ++fly) {
      const double wi = fly ? wd * qinv : wd / qd;
      const double t = pirb::f64_modmul(y, wd, wi, qd);
      CHECK(is_integer(t), "modmul result not an integer: y=%.0f w=%llu q=%llu", y, w, q);
      const i128 exact = (i128)(long long)y * (i128)w;
      CHECK(mod_i128(exact, q) == mod_i128((i128)(long long)t, q), "modmul not congruent: y=%.0f w=%llu q=%llu", y, w, q);
      const double ratio = std::fabs(t) / qd;
      double* worst = fly ? worst_fly : worst_table;
      if (ratio > *worst) *worst = ratio;
      // canonicalisation of the product
      const double c = pirb::f64_canon(t, qd, qinv);
      CHECK(c >= 0.0 && c < qd && is_integer(c) && (u64)c == mod_i128(exact, q), "canon wrong: y=%.0f w=%llu", y, w);
    }
    return 0;
  };
  const double ymax = 281474976710655.0;  // 2^48 - 1
  std::uniform_int_distribution<u64> dw(0, q - 1);
  std::uniform_int_distribution<long long> dy(-(long long)ymax, (long long)ymax);
  std::uniform_int_distribution<long long> dsmall(-9 * (long long)q, 9 * (long long)q);
  for (int i = 0; i < 400000; ++i) {
    if (one((double)dy(rng), dw(rng))) return 1;
    if (one((double)dsmall(rng), dw(rng))) return 1;  // the magnitudes the transforms actually see (< 9q)
  }
  // adversarial: extremes
  for (u64 w : {0ull, 1ull, 2ull, q - 1, q - 2, q / 2, q / 2 + 1})
    for (double y : {0.0, 1.0, -1.0, ymax, -ymax, (double)q, -(double)q, 9.0 * qd, -9.0 * qd, qd - 1.0})
      if (one(y, w)) return 1;
  // adversarial: y*w/q next to a half-integer (the rounding of the quotient estimate is decided by the last bits)
  for (int i = 0; i < 200000; ++i) {
    const u64 w = dw(rng) | 1;
    const u64 m = rng() % (1ull << 30);
    const double target = ((double)m + 0.5) * qd / (double)w;
    if (target >= ymax) continue;
    const double y0 = std::floor(target);
    for (double y : {y0 - 1, y0, y0 + 1, y0 + 2, -(y0), -(y0 + 1)})
      if (one(y, w)) return 1;
  }
  return 0;
}

static ModC make_modc(u64 q, int half_bits, const pirb::hm::Tables& T, std::vector<double2>& fw2,
                            std::vector<double2>& iw2, std::vector<double2>& fin2) {
  ModC m;
  std::memset(&m, 0, sizeof(m));
  m.q = q;
  pirb::hm::barrett_ratio(q, &m.ratio_hi, &m.ratio_lo);
  m.inv_n = T.inv_n;
  m.inv_n_s = T.inv_n_s;
  m.rp = T.rp.data(); m.rps = T.rps.data(); m.irp = T.irp.data(); m.irps = T.irps.data();
  m.qd = (double)q;
  m.qinv = 1.0 / (double)q;
  const size_t N = T.fw.size();
  fw2.resize(N); iw2.resize(N); fin2.resize(N);
  for (size_t i = 0; i < N; ++i) {
    fw2[i] = make_double2(T.fw[i], T.fwi[i]);
    iw2[i] = make_double2(T.iw[i], T.iwi[i]);
    fin2[i] = make_double2(T.fin[i], T.fini[i]);
  }
  m.fw = fw2.data(); m.iw = iw2.data(); m.fin = fin2.data();
  m.fw1 = T.fw.data(); m.iw1 = T.iw.data();
  const u64 ph = pirb::hm::powmod(2, (u64)half_bits, q), p2h = pirb::hm::powmod(2, 2ull * half_bits, q);
  m.pow_h = (double)ph; m.pow_h_i = (double)ph / (double)q;
  m.pow_2h = (double)p2h; m.pow_2h_i = (double)p2h / (double)q;
  return m;
}

// the transforms of pirb_device.cuh, one emulated thread at a time, one pass at a time (a block barrier separates passes)
template <int LOGN, int NT, int S0, int R, class TW>
static void fwd_pass_all(double* d, TW tw, double q) {
  for (int tid = 0; tid < NT; ++tid) pirb::f64_fwd_pass<LOGN, NT, S0, R>(d, tw, q, tid);
}
template <int LOGN, int NT, int S0, int R, class TW>
static void inv_pass_all(double* d, TW tw, double q) {
  for (int tid = 0; tid < NT; ++tid) pirb::f64_inv_pass<LOGN, NT, S0, R>(d, tw, q, tid);
}
template <int LOGN, class TW>
static void forward_emulated(double* d, TW tw, double q) {
  constexpr int NT = ((1 << LOGN) / 8 < 512) ? (1 << LOGN) / 8 : 512;
  constexpr int R0 = ((LOGN - 1) % 3) + 1;
  fwd_pass_all<LOGN, NT, 0, R0>(d, tw, q);
  if constexpr (LOGN > R0) fwd_pass_all<LOGN, NT, R0, 3>(d, tw, q);
  if constexpr (LOGN > R0 + 3) fwd_pass_all<LOGN, NT, R0 + 3, 3>(d, tw, q);
  if constexpr (LOGN > R0 + 6) fwd_pass_all<LOGN, NT, R0 + 6, 3>(d, tw, q);
  if constexpr (LOGN > R0 + 9) fwd_pass_all<LOGN, NT, R0 + 9, 3>(d, tw, q);
}
template <int LOGN, class TW>
static void inverse_emulated(double* d, TW tw, double q) {
  constexpr int NT = ((1 << LOGN) / 8 < 512) ? (1 << LOGN) / 8 : 512;
  constexpr int R0 = ((LOGN - 1) % 3) + 1;
  if constexpr (LOGN > R0 + 9) inv_pass_all<LOGN, NT, R0 + 9, 3>(d, tw, q);
  if constexpr (LOGN > R0 + 6) inv_pass_all<LOGN, NT, R0 + 6, 3>(d, tw, q);
  if constexpr (LOGN > R0 + 3) inv_pass_all<LOGN, NT, R0 + 3, 3>(d, tw, q);
  if constexpr (LOGN > R0) inv_pass_all<LOGN, NT, R0, 3>(d, tw, q);
  inv_pass_all<LOGN, NT, 0, R0>(d, tw, q);
}

template <int LOGN>
static int check_ntt(u64 q, std::mt19937_64& rng) {
  constexpr int N = 1 << LOGN;
  const pirb::hm::Tables T = pirb::hm::build_tables(q, LOGN);
  std::vector<double2> fw2, iw2, fin2;
  const ModC m = make_modc(q, 22, T, fw2, iw2, fin2);
  orc::NttTable ot;
  ot.init(q, LOGN);
  std::vector<u64> x(N), want(N);
  std::uniform_int_distribution<u64> dv(0, q - 1);
  for (int rep = 0; rep < 3; ++rep) {
    for (auto& v : x) v = rep == 0 ? q - 1 : dv(rng);  // all-maximal input first (worst-case growth)
    want = x;
    ot.forward(reinterpret_cast<uint64_t*>(want.data()));
    for (int src = 0; src < 2; ++src) {  // twiddles from the pair table / from the w-only table (w/q formed on the fly)
      std::vector<double> s(N);
      for (int i = 0; i < N; ++i) s[pirb::swz(i)] = pirb::u64_to_f64_exact(x[i]);
      if (src == 0) forward_emulated<LOGN>(s.data(), pirb::TwGlobal{m.fw}, m.qd);
      else forward_emulated<LOGN>(s.data(), pirb::TwShared{m.fw1, m.qinv}, m.qd);
      double growth = 0;
      for (int i = 0; i < N; ++i) {
        const double v = s[pirb::swz(i)];
        CHECK(is_integer(v), "forward output not an integer");
        growth = std::max(growth, std::fabs(v) / m.qd);
        const u64 got = pirb::f64_to_u64_exact(pirb::f64_canon(v, m.qd, m.qinv));
        CHECK(got == want[i], "forward NTT differs from the oracle at %d (q=%llu, N=%d, source %d)", i, q, N, src);
      }
      CHECK(growth < 9.0, "forward growth %.2f q exceeds the documented bound", growth);
      // inverse of the (lazy, uncanonicalised) forward output must give the input back
      if (src == 0) inverse_emulated<LOGN>(s.data(), pirb::TwGlobal{m.iw}, m.qd);
      else inverse_emulated<LOGN>(s.data(), pirb::TwShared{m.iw1, m.qinv}, m.qd);
      for (int i = 0; i < N; ++i) {
        u64 word;
        std::memcpy(&word, &s[pirb::swz(i)], 8);
        const u64 got = pirb::eng_store_inv<pirb::ENG_FP64>(word, i, m);
        CHECK(got == x[i], "inverse NTT does not return the input at %d (q=%llu, N=%d, source %d)", i, q, N, src);
      }
    }
    // inverse alone against the oracle's inverse
    std::vector<u64> y(N), wanti(N);
    for (auto& v : y) v = dv(rng);
    wanti = y;
    ot.inverse(reinterpret_cast<uint64_t*>(wanti.data()));
    std::vector<double> s(N);
    for (int i = 0; i < N; ++i) s[pirb::swz(i)] = pirb::u64_to_f64_exact(y[i]);
    inverse_emulated<LOGN>(s.data(), pirb::TwGlobal{m.iw}, m.qd);
    for (int i = 0; i < N; ++i) {
      u64 word;
      std::memcpy(&word, &s[pirb::swz(i)], 8);
      CHECK(pirb::eng_store_inv<pirb::ENG_FP64>(word, i, m) == wanti[i], "inverse NTT differs from the oracle at %d", i);
    }
  }
  return 0;
}

static int check_mac_chains(u64 q, int half_bits, std::mt19937_64& rng) {
  const pirb::hm::Tables T = pirb::hm::build_tables(q, 11);
  std::vector<double2> fw2, iw2, fin2;
  const ModC m = make_modc(q, half_bits, T, fw2, iw2, fin2);
  const unsigned max_terms = 1u << std::min(14, 51 - 2 * half_bits);
  std::uniform_int_distribution<u64> dv(0, q - 1);
  for (int rep = 0; rep < 20; ++rep) {
    pirb::Acc<pirb::MAC_FP64> af;
    pirb::Acc<pirb::MAC_INT24> ai;
    pirb::Acc<pirb::MAC_WIDE>* unused = nullptr;  // (its carry chain is PTX; covered on the GPU)
    (void)unused;
    u128 exact = 0;
    for (unsigned i = 0; i < max_terms; ++i) {
      const u64 a = rep == 0 ? q - 1 : dv(rng), b = rep == 0 ? q - 1 : dv(rng);  // all-maximal chain first
      af.mac(pirb::Opnd<pirb::MAC_FP64>(a, half_bits), pirb::Opnd<pirb::MAC_FP64>(b, half_bits));
      if (q < (1ull << 48) && i < pirb::PIRB_SMALL_MAX_TERMS)
        ai.mac(pirb::Opnd<pirb::MAC_INT24>(a, 24), pirb::Opnd<pirb::MAC_INT24>(b, 24));
      exact += (u128)a * b;
    }
    CHECK(is_integer(af.s0) && is_integer(af.sk) && is_integer(af.s2) && af.sk < 9007199254740992.0,
          "FP64 partial sums left the exact range");
    CHECK(af.reduce(m, half_bits) == (u64)(exact % q), "FP64 Karatsuba chain differs (q=%llu, h=%d)", q, half_bits);
    if (q < (1ull << 48)) CHECK(ai.reduce(m, 24) == (u64)(exact % q), "24-bit Karatsuba chain differs (q=%llu)", q);
    CHECK(pirb::barrett128((u64)exact, (u64)(exact >> 64), q, m.ratio_hi, m.ratio_lo) == (u64)(exact % q), "barrett128");
  }
  for (int i = 0; i < 200000; ++i) {
    const u64 x = rng(), w = dv(rng);
    CHECK(pirb::shoup(x, w, pirb::hm::shoup(w, q), q) == (u64)((u128)x * w % q), "shoup");
    CHECK(pirb::barrett64(x, q, m.ratio_hi) == x % q, "barrett64");
    const u64 v = x >> 12;
    CHECK(pirb::f64_to_u64_exact(pirb::u64_to_f64_exact(v)) == v, "u64 <-> double conversion");
  }
  return 0;
}

static int check_galois(std::mt19937_64& rng) {
  const int logn = 12, N = 1 << logn;
  const u64 q = 0xffffee001ull;
  std::vector<u64> in(N), want(N);
  for (auto& v : in) v = rng() % q;
  for (uint32_t g : {3u, 5u, (uint32_t)N + 1, (uint32_t)N / 2 + 1, 2u * N - 1}) {
    orc::apply_galois_poly(reinterpret_cast<const uint64_t*>(in.data()), N, logn, g, orc::Modulus(q),
                           reinterpret_cast<uint64_t*>(want.data()));
    uint32_t ginv = g;
    for (int i = 0; i < 5; ++i) ginv *= 2 - g * ginv;  // Newton iteration modulo a power of two
    ginv &= 2 * N - 1;
    for (int n = 0; n < N; ++n)
      CHECK(pirb::galois_gather(in.data(), n, ginv, N, q) == want[n], "galois gather differs (g=%u, n=%d)", g, n);
  }
  return 0;
}

// The launch plan of the tensor-core batched scan (tc_plan.h) for every shape it can be asked for: each plan it accepts
// must be launchable and exact, it must take the widest query tile that fits, and it may refuse only when not even the
// narrowest tile fits.  The plans of the benchmark workloads are pinned: those scans launch exactly as they did before
// the plan was factored out.
static int check_tc_plans() {
  const uint32_t A = pirb::TC_A_STAGE_BYTES, budget = pirb::TC_SMEM_BUDGET;
  long accepted = 0;
  for (uint32_t nb : {5u, 6u}) {
    const uint32_t fixed = pirb::TC_MAX_ACC * 16 * 128 * 8 * (nb == 5 ? 1 : 2) + 1024;
    const uint32_t dimL_max = nb == 5 ? 2048 : 1280;  // kch 16 / 10: the last B operand of qt 8 that fits
    for (int req : {8, 16, 24}) {
      for (uint32_t dimL = 1; dimL <= 33000; ++dimL) {
        pirb::TcPlan prev = {};
        bool prev_ok = true;
        for (uint32_t nq = 1; nq <= 64; ++nq) {
          pirb::TcPlan p;
          const bool ok = pirb::tc_plan(nb, dimL, nq, req, &p);
          CHECK(ok == (dimL <= dimL_max), "plan existence (nb %u, dimL %u, %u queries, qt %d): %d", nb, dimL, nq, req, ok);
          if (!ok) continue;
          ++accepted;
          CHECK(prev_ok, "a plan for %u queries but none for fewer (nb %u, dimL %u)", nq, nb, dimL);
          CHECK(p.smem <= budget && p.stages >= 2 && p.stages <= 8, "shared memory %u B, %u stages (nb %u, dimL %u, %u q)",
                p.smem, p.stages, nb, dimL, nq);
          CHECK(p.qt % 8 == 0 && p.qt >= 8 && (int)p.qt <= std::max(8, req / 8 * 8), "qt %u for requested %d", p.qt, req);
          CHECK(p.n_cols == p.qt * 2 * nb && p.n_cols % 16 == 0 && p.n_cols <= 256, "MMA N %u (nb %u, qt %u)", p.n_cols, nb,
                p.qt);
          CHECK(p.n_qt * p.qt >= nq && (p.n_qt - 1) * p.qt < nq, "%u tiles of %u queries for %u queries", p.n_qt, p.qt, nq);
          CHECK(p.Kp >= dimL && p.Kp % 16 == 0 && p.Kp < dimL + 16 && p.kch * 128 >= p.Kp && (p.kch - 1) * 128 < p.Kp,
                "K geometry Kp %u kch %u for dimL %u", p.Kp, p.kch, dimL);
          CHECK((uint64_t)dimL * 255 * 255 < (1ull << 31), "s32 accumulator bound at dimL %u", dimL);
          const uint32_t b_buf = p.kch * p.n_cols * 128;
          CHECK(p.smem == p.stages * A + p.b_bufs * b_buf + fixed, "shared memory accounting");
          CHECK(p.b_bufs == ((2 * b_buf + fixed + 4 * A <= budget) ? 2u : 1u), "b_bufs %u (nb %u, dimL %u, qt %u)", p.b_bufs,
                nb, dimL, p.qt);
          CHECK(p.stages == std::min<uint32_t>(8, (budget - fixed - p.b_bufs * b_buf) / A), "A ring depth");
          // widest tile: the next wider one allowed by the request and the query count would not fit
          const uint32_t cap = std::min(std::min((nq + 7) / 8 * 8, nb == 5 ? 24u : 16u), (uint32_t)std::max(8, req / 8 * 8));
          if (p.qt < cap)
            CHECK(p.kch * (p.qt + 8) * 2 * nb * 128 + fixed + 2 * A > budget, "qt %u chosen although %u fits (dimL %u)",
                  p.qt, p.qt + 8, dimL);
          else
            CHECK(p.qt == cap, "qt %u above the cap %u", p.qt, cap);
          if (nq > 1) CHECK(p.qt >= prev.qt, "qt shrinks from %u to %u as queries grow", prev.qt, p.qt);
          prev = p;
          prev_ok = ok;
        }
      }
    }
  }
  // the shapes that used to be refused at launch: a narrower tile now
  pirb::TcPlan p;
  CHECK(pirb::tc_plan(5, 1024, 16, 16, &p) && p.qt == 16, "nb 5 dimL 1024");
  CHECK(pirb::tc_plan(5, 1025, 9, 16, &p) && p.qt == 8 && p.n_qt == 2, "nb 5 dimL 1025");
  CHECK(pirb::tc_plan(5, 640, 24, 24, &p) && p.qt == 24, "nb 5 dimL 640 qt 24");
  CHECK(pirb::tc_plan(5, 641, 24, 24, &p) && p.qt == 16 && p.n_qt == 2, "nb 5 dimL 641 qt 24");
  CHECK(pirb::tc_plan(6, 640, 16, 16, &p) && p.qt == 16, "nb 6 dimL 640");
  CHECK(pirb::tc_plan(6, 641, 9, 16, &p) && p.qt == 8 && p.n_qt == 2, "nb 6 dimL 641");
  CHECK(!pirb::tc_plan(6, 1281, 4, 16, &p) && !pirb::tc_plan(5, 2049, 4, 16, &p), "beyond the narrowest tile");
  // benchmark workloads (default PIRB_TC_QT): configs[3] (N=4096, dims [333, 332]) with 8 queries on one GPU and 16 / 64
  // per scan on several; configs[4] d=2 (N=4096, [665, 664]) with 8 and 16; configs[2] (N=8192, [235, 235]) with 4..16
  struct Want { uint32_t nb, dimL, nq, qt, n_qt, kch, b_bufs, stages, smem; };
  const Want bench[] = {{5, 332, 8, 8, 1, 3, 2, 8, 226304},  {5, 332, 16, 16, 1, 3, 2, 4, 222208},
                        {5, 332, 64, 16, 4, 3, 2, 4, 222208}, {5, 664, 8, 8, 1, 6, 2, 4, 222208},
                        {5, 664, 16, 16, 1, 6, 1, 4, 222208}, {6, 235, 4, 8, 1, 2, 2, 7, 230400},
                        {6, 235, 8, 8, 1, 2, 2, 7, 230400},   {6, 235, 16, 16, 1, 2, 2, 4, 230400}};
  for (const Want& w : bench) {
    CHECK(pirb::tc_plan(w.nb, w.dimL, w.nq, 16, &p), "bench plan missing (dimL %u, %u queries)", w.dimL, w.nq);
    CHECK(p.qt == w.qt && p.n_qt == w.n_qt && p.kch == w.kch && p.b_bufs == w.b_bufs && p.stages == w.stages &&
              p.smem == w.smem,
          "bench plan changed (dimL %u, %u queries): qt %u n_qt %u kch %u b_bufs %u stages %u smem %u", w.dimL, w.nq, p.qt,
          p.n_qt, p.kch, p.b_bufs, p.stages, p.smem);
  }
  std::printf("tensor-core scan plans: %ld accepted shapes launchable and exact, benchmark plans unchanged\n", accepted);
  return 0;
}

int main() {
  std::mt19937_64 rng(2024);
  if (check_tc_plans()) return 1;
  // BFVDefault primes of N=4096 / N=8192, the 24-bit-plain config's moduli are the same; plus a 44-bit prime (the
  // largest the FP64 engine accepts)
  std::vector<u64> moduli;
  for (u64 v : orc::bfv_default_coeff_modulus(4096)) moduli.push_back(v);
  for (u64 v : orc::bfv_default_coeff_modulus(8192)) moduli.push_back(v);
  u64 p44 = (1ull << 44) - (1ull << 15) + 1;
  while (!(pirb::hm::is_prime(p44) && p44 % (2 * 16384) == 1)) p44 -= 2 * 16384;
  moduli.push_back(p44);
  double worst_table = 0, worst_fly = 0;
  for (u64 q : moduli)
    if (check_modmul(q, rng, &worst_table, &worst_fly)) return 1;
  std::printf("f64_modmul exact on %zu moduli; max |t|/q = %.4f (table companion), %.4f (on-the-fly companion)\n",
              moduli.size(), worst_table, worst_fly);
  CHECK(worst_table <= 0.54 && worst_fly <= 0.57, "product magnitude bound violated");
  for (u64 q : moduli) {
    int bits = 0;
    while ((q >> bits) != 0) ++bits;
    if (check_mac_chains(q, (bits + 1) / 2, rng)) return 1;
  }
  std::printf("multiply-accumulate chains exact at their maximum length\n");
  for (u64 q : orc::bfv_default_coeff_modulus(4096))
    if (check_ntt<12>(q, rng)) return 1;
  if (check_ntt<11>(orc::bfv_default_coeff_modulus(4096)[0], rng)) return 1;
  if (check_ntt<13>(orc::bfv_default_coeff_modulus(8192)[0], rng)) return 1;
  if (check_ntt<13>(orc::bfv_default_coeff_modulus(8192)[4], rng)) return 1;
  if (check_ntt<14>(p44, rng)) return 1;
  std::printf("device NTT passes (pair-table and shared-table twiddles) match the oracle for N = 2048 .. 16384\n");
  if (check_galois(rng)) return 1;
  std::printf("DEVICE_MATH_HOST_TEST_OK\n");
  return 0;
}
