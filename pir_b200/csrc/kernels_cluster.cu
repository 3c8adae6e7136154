// kernels_cluster.cu — one expansion level (Galois automorphism + key switch + SealPIR butterfly) in ONE launch.
//
// Reference: server.cpp:123-141 per tree node; Evaluator::apply_galois_inplace -> switch_key_inplace (SURVEY A.4-A.6).
// A thread-block cluster of 2(k+1) CTAs owns one node.  CTA rank r works on key-level modulus I = r/2 and key
// component c = r%2:
//   phase 1  the pair (I,0),(I,1) splits the k RNS digits: sigma_g(c1) digit J (J%2 == c) is re-reduced mod m_I and
//            forward-transformed in shared memory;
//   phase 2  acc[c][I] = sum_J dig[I][J] (.) key[J][c][I]  — own digits from local shared memory, the partner's through
//            distributed shared memory — then the inverse transform, all without leaving the SM;
//   phase 3  CTAs with I < k mod-down their polynomial by P (reading acc[c][P] from the (k,c) CTA's shared memory), add
//            sigma_g(c0) and write the even/odd children of the node.
// Compared with the three-kernel path (k_ks_digits, k_ks_mac_intt, k_ks_combine) the digit and accumulator
// polynomials never touch global memory and a tree level costs one launch instead of three.
#include <cooperative_groups.h>

#include <algorithm>
#include <cstdlib>

#include <type_traits>

#include "kernels.cuh"
#include "pirb_device.cuh"

namespace cg = cooperative_groups;

namespace pirb {

template <int LOGN>
struct CCfg {
  static constexpr int N = 1 << LOGN;
  static constexpr int NT = (N / 8 < 512) ? N / 8 : 512;
};

__device__ __forceinline__ u64 mod_down_c(u64 a, u64 last, const DevParams& P, int j, u64 Pq) {
  const ModC& m = P.m[j];
  u64 l = last + P.half_P;
  l = l >= Pq ? l - Pq : l;
  u64 r = submod(barrett64(l, m.q, m.ratio_hi), P.half_P_mod[j], m.q);
  return shoup(submod(a, r, m.q), P.inv_P[j], P.inv_P_s[j], m.q);
}

// The key of the node's query: the launch's key, or with a per-query key table that query's client's key.  The first
// generation reads it where it is used (a register holding it across the phases costs spills in <12,2,*>); the second
// keeps it in a register (fewer spills there).
#define PIRB_QKEY \
  (L.key_tab ? reinterpret_cast<const u64*>(__ldg(reinterpret_cast<const unsigned long long*>(L.key_tab) + qi)) : key_arg)
template <int LOGN, int ENG, int MODE>
__global__ void __launch_bounds__(CCfg<LOGN>::NT, (LOGN <= 12 ? 2 : 1))
k_ks_level_cluster(const __grid_constant__ DevParams P, u64* __restrict__ work, const LevelArgs L,
                   const u64* __restrict__ key_arg, int mode) {
  constexpr int N = CCfg<LOGN>::N, NT = CCfg<LOGN>::NT;
  extern __shared__ u64 smem[];
  cg::cluster_group cluster = cg::this_cluster();
  const int tid = threadIdx.x;
  const int k = P.k;
  const int csize = 2 * (k + 1);
  const unsigned rank = cluster.block_rank();
  const int I = rank >> 1, c = rank & 1;
  const u32 z = blockIdx.x / csize;  // node
  const u32 kk = z & ((1u << L.j) - 1);
  const u32 tq = z >> L.j;
  const u32 ti = tq % L.n_trees, qi = tq / L.n_trees;
  const u64 ctL = (u64)2 * k * N;
  const u64* src = work + qi * L.q_stride + L.src_off[ti] + kk * ctL;
  const ModC& mI = P.m[I];
  const int nd = (k + 1) / 2;  // digit buffers per CTA
  u64* A = smem + (size_t)nd * N;
  // FP64 engine, N <= 4096: the twiddle table of the running transform is staged in shared memory by one bulk
  // asynchronous copy (forward table while the digits are gathered, inverse table while the key products are
  // formed), so no butterfly pass waits on an L2 round trip for its twiddles
  constexpr bool TWS = (ENG == ENG_FP64) && (LOGN <= 12);
  double* TWb = reinterpret_cast<double*>(A + N);
  u64* twbar = A + 2 * (size_t)N;
  if constexpr (TWS) {
    if (tid == 0) {
      mbar_init(twbar, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
      mbar_expect_tx(twbar, N * 8);
      bulk_g2s_plain(TWb, mI.fw1, N * 8, twbar);
    }
  }
#define PIRB_STAMP(slot)                                                                   \
  do {                                                                                     \
    if (L.dbg && tid == 0) {                                                               \
      u64 t_;                                                                              \
      if (((slot) == 0 || (slot) == 7) && !L.dbg_clock) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); \
      else t_ = clock64();                                                                 \
      L.dbg[(u64)blockIdx.x * 8 + (slot)] = t_;                                            \
    }                                                                                      \
  } while (0)
  PIRB_STAMP(0);
  asm volatile("griddepcontrol.launch_dependents;");  // the next level may start its own prologue now
  // Prologue: pull everything this CTA will read from global memory into L2 now (one 128-byte line per prefetch), so
  // the key limbs of phase 2 and the source polynomials of phases 1 and 3 are L2 hits when they are needed.
  {
    constexpr int LINES = N * 8 / 128;  // lines per polynomial
    for (int J = 0; J < k; ++J) {
      const char* kp = reinterpret_cast<const char*>(PIRB_QKEY + ((u64)(J * 2 + c) * (k + 1) + I) * N);
      for (int l = tid; l < LINES; l += NT) asm volatile("prefetch.global.L2 [%0];" ::"l"(kp + (size_t)l * 128));
    }
    // Programmatic dependent launch: everything above (key prefetch, index math) may overlap the tail of the previous
    // level's kernel; from here on we read what it wrote.
    asm volatile("griddepcontrol.wait;" ::: "memory");
    for (int J = c; J < k; J += 2) {
      const char* sp = reinterpret_cast<const char*>(src + (u64)(k + J) * N);
      for (int l = tid; l < LINES; l += NT) asm volatile("prefetch.global.L2 [%0];" ::"l"(sp + (size_t)l * 128));
    }
    if (I < k) {
      const char* sp = reinterpret_cast<const char*>(src + (u64)(c * k + I) * N);
      for (int l = tid; l < LINES; l += NT) asm volatile("prefetch.global.L2 [%0];" ::"l"(sp + (size_t)l * 128));
    }
  }

  // ---- phase 1: my digits ----
  for (int J = c; J < k; J += 2) {
    u64* D = smem + (size_t)(J >> 1) * N;
    const u64* c1 = src + (u64)(k + J) * N;
    const u64 qJ = P.m[J].q;
    const bool need_reduce = qJ > mI.q;
#pragma unroll
    for (int i = tid; i < N; i += NT) {
      u64 v = galois_gather(c1, i, L.ginv, N, qJ);
      if (need_reduce) v = barrett64(v, mI.q, mI.ratio_hi);
      D[swz(i)] = eng_load<ENG>(v);
    }
    __syncthreads();
    PIRB_STAMP(1);
    if constexpr (TWS) {
      mbar_wait(twbar, 0);
      f64_forward_all<LOGN, NT>(reinterpret_cast<double*>(D), TwShared{TWb, mI.qinv}, mI.qd, tid);
    } else {
      eng_forward<LOGN, NT, ENG>(D, mI, tid);
    }
    PIRB_STAMP(2);
    // FP64 engine: the transform's output (integer-valued, below 9q in magnitude) goes into the key products as it is —
    // f64_modmul is exact for |y| < 2^48, so a canonicalisation pass over the digit would be wasted work
    if constexpr (ENG != ENG_FP64) {
#pragma unroll
      for (int i = tid; i < N; i += NT) D[swz(i)] = eng_store_fwd<ENG>(D[swz(i)], mI);
    }
  }
  if constexpr (TWS) {
    // every forward pass has ended with a block barrier: the table buffer is free for the inverse twiddles.  A CTA
    // without digits (c = 1 when k = 1) has not waited for the forward table yet; its copy must have landed before
    // the barrier is armed again and the buffer rewritten (otherwise two copies race into it and the second arrival
    // lands on a phase that is still pending).
    if (tid == 0) {
      mbar_wait(twbar, 0);
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      mbar_expect_tx(twbar, N * 8);
      bulk_g2s_plain(TWb, mI.iw1, N * 8, twbar);
    }
  }
  PIRB_STAMP(3);
  cluster.sync();
  PIRB_STAMP(4);

  // ---- phase 2: MAC with the key, inverse transform ----
  {
    const u64* peer = cluster.map_shared_rank(smem, rank ^ 1);
    const int hb = P.half_bits;
    // four coefficients per thread at a time; for every digit all operand loads (shared / distributed shared /
    // global) are issued before the first multiply so their latencies overlap
    constexpr int CH = 4;
    if constexpr (ENG == ENG_FP64) {
      // k <= 8 terms: one exact FP64 modular product per term (digit (.) key), summed and canonicalised once.
      // The key limb's w/q companion is formed on the fly (kv * (1/q)); its 2^-51 relative error keeps the
      // quotient estimate within 0.51 of the true value, so |product| <= 0.54 q as for table constants.
      const double qd = mI.qd, qinv = mI.qinv;
#pragma unroll 1
      for (int i0 = tid; i0 < N; i0 += CH * NT) {
        double acc[CH];
        int si[CH];
#pragma unroll
        for (int e = 0; e < CH; ++e) { si[e] = swz(i0 + e * NT); acc[e] = 0.0; }
#pragma unroll 2
        for (int J = 0; J < k; ++J) {
          const u64* buf = (((J & 1) == c) ? smem : peer) + (size_t)(J >> 1) * N;
          const u64* kp = PIRB_QKEY + ((u64)(J * 2 + c) * (k + 1) + I) * N + i0;
          u64 dv[CH], kv[CH];
#pragma unroll
          for (int e = 0; e < CH; ++e) {
            dv[e] = buf[si[e]];
            kv[e] = __ldg(kp + e * NT);
          }
#pragma unroll
          for (int e = 0; e < CH; ++e) {
            const double kd = u64_to_f64_exact(kv[e]);
            const double t = f64_modmul(__longlong_as_double((long long)dv[e]), kd, __dmul_rn(kd, qinv), qd);
            acc[e] = __dadd_rn(acc[e], t);
          }
        }
#pragma unroll
        for (int e = 0; e < CH; ++e) A[si[e]] = (u64)__double_as_longlong(f64_canon(acc[e], qd, qinv));
      }
    } else {
#pragma unroll 1
      for (int i0 = tid; i0 < N; i0 += CH * NT) {
        Acc<MODE> acc[CH];
        int si[CH];
#pragma unroll
        for (int e = 0; e < CH; ++e) si[e] = swz(i0 + e * NT);
#pragma unroll 1
        for (int J = 0; J < k; ++J) {
          const u64* buf = (((J & 1) == c) ? smem : peer) + (size_t)(J >> 1) * N;
          const u64* kp = PIRB_QKEY + ((u64)(J * 2 + c) * (k + 1) + I) * N + i0;
          u64 dv[CH], kv[CH];
#pragma unroll
          for (int e = 0; e < CH; ++e) {
            dv[e] = buf[si[e]];
            kv[e] = __ldg(kp + e * NT);
          }
#pragma unroll
          for (int e = 0; e < CH; ++e) acc[e].mac(Opnd<MODE>(dv[e], hb), Opnd<MODE>(kv[e], hb));
        }
#pragma unroll
        for (int e = 0; e < CH; ++e) A[si[e]] = eng_load<ENG>(acc[e].reduce(mI, hb));
      }
    }
    __syncthreads();
    PIRB_STAMP(5);
    if constexpr (TWS) {
      mbar_wait(twbar, 1);
      f64_inverse_all<LOGN, NT>(reinterpret_cast<double*>(A), TwShared{TWb, mI.qinv}, mI.qd, tid);
    } else {
      eng_inverse<LOGN, NT, ENG>(A, mI, tid);
    }
    if (!(L.dbg_clock & 2)) PIRB_STAMP(6);
    if (I == k) {
      // special-prime accumulator: hand it to the readers through global memory.  Distributed shared memory moves
      // ~21 B/clk per source SM and each of these CTAs feeds k readers; the same 8 B per coefficient through L2 is
      // several times faster.  barrier.cluster (release/acquire) orders these stores before the readers' loads.
      u64* xo = L.xch + ((u64)z * 2 + c) * N;
#pragma unroll
      for (int i = tid; i < N; i += NT) xo[i] = eng_finish_inv_native<ENG>(A[swz(i)], i, mI);
    } else {
#pragma unroll
      for (int i = tid; i < N; i += NT) A[swz(i)] = eng_finish_inv_native<ENG>(A[swz(i)], i, mI);
      if constexpr (TWS) {
        // the twiddle buffer is free again: stage this CTA's source polynomial there (coalesced loads), so that the
        // Galois gather sigma_g(c0) of phase 3 is a shared-memory permutation instead of scattered global sectors
        const u64* sp = src + (u64)(c * k + I) * N;
        u64* SB = reinterpret_cast<u64*>(TWb);
#pragma unroll
        for (int i = tid; i < N; i += NT) SB[i] = sp[i];
      }
    }
  }
  cluster.sync();
  if (L.dbg_clock & 2) PIRB_STAMP(6);  // PIRB_STAMP_CLOCK=3: slot 6 after the barrier, to split the tail

  // ---- phase 3: mod-down by P, add sigma_g(c0), expansion butterfly ----
  if (I < k) {
    const int j = I;
    const u64 q = mI.q, Pq = P.m[k].q;
    const u64* lastA = L.xch + ((u64)z * 2 + c) * N;
    const u64* SB = reinterpret_cast<const u64*>(TWb);
    u64* dstE = work + qi * L.q_stride + L.dst_off[ti] + kk * ctL;
    const u64* sp = src + (u64)(c * k + j) * N;
    const u32 s1 = (2 * N - (1u << L.j)) & (2 * N - 1);
    // Source and destination live in the same workspace, so the compiler must keep every load behind the previous
    // element's stores; gather all operands of CH elements first (distributed shared memory, shared memory, global)
    // and only then compute and store, so their latencies overlap instead of adding up.
    constexpr int CH = 4;
#pragma unroll 1
    for (int i0 = tid; i0 < N; i0 += CH * NT) {
      u64 la[CH], av[CH], pv[CH], gv[CH];
#pragma unroll
      for (int e = 0; e < CH; ++e) {
        const int i = i0 + e * NT, si = swz(i);
        la[e] = __ldcg(lastA + i);
        av[e] = A[si];
        if constexpr (TWS) {
          gv[e] = (c == 0) ? galois_gather(SB, i, L.ginv, N, q) : 0;
          pv[e] = (mode == 1) ? 0 : SB[i];
        } else {
          gv[e] = (c == 0) ? galois_gather(sp, i, L.ginv, N, q) : 0;
          pv[e] = (mode == 1) ? 0 : sp[i];
        }
      }
#pragma unroll
      for (int e = 0; e < CH; ++e) {
        const int i = i0 + e * NT;
        u64 c0;
        if constexpr (ENG == ENG_FP64) {
          // mod-down by P on the FP64 pipe: ((a - ((l + P/2 mod P) mod q - P/2 mod q)) * P^-1) mod q
          const double qd = mI.qd;
          double l = __dadd_rn(__longlong_as_double((long long)la[e]), P.half_P_d);
          l = l >= P.m[k].qd ? __dadd_rn(l, -P.m[k].qd) : l;
          const double r = f64_submod(f64_canon(l, qd, mI.qinv), P.half_P_mod_d[j], qd);
          const double dd = f64_submod(__longlong_as_double((long long)av[e]), r, qd);
          double md = f64_modmul(dd, P.inv_P_d[j], P.inv_P_di[j], qd);
          md = md < 0.0 ? __dadd_rn(md, qd) : md;
          c0 = f64_to_u64_exact(md);
        } else {
          c0 = mod_down_c(av[e], la[e], P, j, Pq);
        }
        if (c == 0) c0 = addmod(gv[e], c0, q);
        if (mode == 1) {
          dstE[(u64)(c * k + j) * N + i] = c0;
        } else {
          const u64 p = pv[e];
          dstE[(u64)(c * k + j) * N + i] = addmod(p, c0, q);
          const u32 r = i + s1;
          u64 d = submod(p, c0, q);
          if (r & N) d = negmod(d, q);
          (dstE + ((u64)ctL << L.j))[(u64)(c * k + j) * N + (r & (N - 1))] = d;
        }
      }
    }
  }
  PIRB_STAMP(7);
  // no CTA's shared memory is read remotely after the second cluster barrier (the partner's digit reads of phase 2
  // are complete, the special-prime accumulators travel through global memory), so every CTA may exit on its own
}

// ---------------------------------------------------------------------------------------------------------------
// Second generation for the wide levels (FP64 engine, N <= 4096, all k digits in one CTA's shared memory): a cluster of
// k+1 CTAs per node, CTA I owning key-level modulus I for BOTH key components.  It transforms all k digits itself
// (no distributed-shared-memory reads, no cluster barrier before the key products; consecutive transforms share one
// block barrier per pass), forms acc[0][I] and acc[1][I] in place, inverse-transforms both, and after the single
// cluster barrier mod-downs both components.  Per node: (k+1) CTAs x (k forward + 2 inverse) transforms — the same
// arithmetic as the first generation in half as many CTAs, with fewer barriers and no canonicalisation pass.
// ---------------------------------------------------------------------------------------------------------------
template <int LOGN, int K>
__global__ void __launch_bounds__(CCfg<LOGN>::NT, 2)
k_ks_level_cluster2(const __grid_constant__ DevParams P, u64* __restrict__ work, const LevelArgs L,
                    const u64* __restrict__ key_arg, int mode) {
  constexpr int N = CCfg<LOGN>::N, NT = CCfg<LOGN>::NT;
  constexpr int NB = K < 2 ? 2 : K;  // buffers: the k digits; two accumulators live in the first two afterwards
  extern __shared__ u64 smem[];
  cg::cluster_group cluster = cg::this_cluster();
  const int tid = threadIdx.x;
  constexpr int k = K;
  const int I = (int)cluster.block_rank();
  const u32 z = blockIdx.x / (k + 1);  // node
  const u32 kk = z & ((1u << L.j) - 1);
  const u32 tq = z >> L.j;
  const u32 ti = tq % L.n_trees, qi = tq / L.n_trees;
  const u64* __restrict__ key = L.key_tab ? L.key_tab[qi] : key_arg;  // this query's client
  const u64 ctL = (u64)2 * k * N;
  const u64* src = work + qi * L.q_stride + L.src_off[ti] + kk * ctL;
  const ModC& mI = P.m[I];
  const double qd = mI.qd, qinv = mI.qinv;
  double* TWb = reinterpret_cast<double*>(smem + (size_t)NB * N);
  u64* twbar = smem + (size_t)(NB + 1) * N;
  if (tid == 0) {
    mbar_init(twbar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    mbar_expect_tx(twbar, N * 8);
    bulk_g2s_plain(TWb, mI.fw1, N * 8, twbar);
  }
  asm volatile("griddepcontrol.launch_dependents;");
  {
    constexpr int LINES = N * 8 / 128;
    for (int J = 0; J < k; ++J)
      for (int c = 0; c < 2; ++c) {
        const char* kp = reinterpret_cast<const char*>(key + ((u64)(J * 2 + c) * (k + 1) + I) * N);
        for (int l = tid; l < LINES; l += NT) asm volatile("prefetch.global.L2 [%0];" ::"l"(kp + (size_t)l * 128));
      }
    asm volatile("griddepcontrol.wait;" ::: "memory");
  }
  // ---- phase 1: all digits of sigma_g(c1), re-reduced mod m_I, forward transforms ----
#pragma unroll
  for (int J = 0; J < k; ++J) {
    u64* D = smem + (size_t)J * N;
    const u64* c1 = src + (u64)(k + J) * N;
    const u64 qJ = P.m[J].q;
    const bool need_reduce = qJ > mI.q;
    // the automorphism as a SCATTER into shared memory: coalesced global reads of a[i], destination slot i*g mod N
    // with the sign of floor(i*g / N)'s parity (sigma_g(a)[i*g mod N] = +-a[i]; the same map galois_gather inverts)
#pragma unroll
    for (int i = tid; i < N; i += NT) {
      u64 v = c1[i];
      const u32 t = ((u32)i * L.g) & (2 * N - 1);
      if (t & N) v = negmod(v, qJ);
      if (need_reduce) v = barrett64(v, mI.q, mI.ratio_hi);
      D[swz(t & (N - 1))] = eng_load<ENG_FP64>(v);
    }
  }
  __syncthreads();
  mbar_wait(twbar, 0);
  {
    constexpr int R0 = ((LOGN - 1) % 3) + 1;
    const TwShared tw{TWb, qinv};
    auto pass_all = [&](auto s0, auto r) {
      constexpr int S0 = decltype(s0)::value, R = decltype(r)::value;
#pragma unroll
      for (int J = 0; J < k; ++J) f64_fwd_pass<LOGN, NT, S0, R>(reinterpret_cast<double*>(smem + (size_t)J * N), tw, qd, tid);
      __syncthreads();
    };
    pass_all(std::integral_constant<int, 0>{}, std::integral_constant<int, R0>{});
    if constexpr (LOGN > R0) pass_all(std::integral_constant<int, R0>{}, std::integral_constant<int, 3>{});
    if constexpr (LOGN > R0 + 3) pass_all(std::integral_constant<int, R0 + 3>{}, std::integral_constant<int, 3>{});
    if constexpr (LOGN > R0 + 6) pass_all(std::integral_constant<int, R0 + 6>{}, std::integral_constant<int, 3>{});
    if constexpr (LOGN > R0 + 9) pass_all(std::integral_constant<int, R0 + 9>{}, std::integral_constant<int, 3>{});
  }
  if (tid == 0) {  // the table buffer is free: inverse twiddles travel while the key products are formed
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    mbar_expect_tx(twbar, N * 8);
    bulk_g2s_plain(TWb, mI.iw1, N * 8, twbar);
  }
  // ---- phase 2: acc[c] = sum_J digit_J (.) key[J][c][I] for both components, in place ----
  {
    constexpr int CH = 4;
#pragma unroll 1
    for (int i0 = tid; i0 < N; i0 += CH * NT) {
      double a0[CH], a1[CH];
      int si[CH];
#pragma unroll
      for (int e = 0; e < CH; ++e) { si[e] = swz(i0 + e * NT); a0[e] = 0.0; a1[e] = 0.0; }
#pragma unroll
      for (int J = 0; J < k; ++J) {
        const u64* D = smem + (size_t)J * N;
        const u64* kp0 = key + ((u64)(J * 2 + 0) * (k + 1) + I) * N + i0;
        const u64* kp1 = key + ((u64)(J * 2 + 1) * (k + 1) + I) * N + i0;
        u64 dv[CH], k0[CH], k1[CH];
#pragma unroll
        for (int e = 0; e < CH; ++e) {
          dv[e] = D[si[e]];
          k0[e] = __ldg(kp0 + e * NT);
          k1[e] = __ldg(kp1 + e * NT);
        }
#pragma unroll
        for (int e = 0; e < CH; ++e) {
          const double y = __longlong_as_double((long long)dv[e]);
          const double kd0 = u64_to_f64_exact(k0[e]), kd1 = u64_to_f64_exact(k1[e]);
          a0[e] = __dadd_rn(a0[e], f64_modmul(y, kd0, __dmul_rn(kd0, qinv), qd));
          a1[e] = __dadd_rn(a1[e], f64_modmul(y, kd1, __dmul_rn(kd1, qinv), qd));
        }
      }
      // sums of k products of magnitude <= 0.54 q each: the inverse transform's butterflies only need |v| < 2^48 and add
      // at most 0.54 q per stage, so the accumulators go in as they are (no canonicalisation pass)
#pragma unroll
      for (int e = 0; e < CH; ++e) {
        smem[si[e]] = (u64)__double_as_longlong(a0[e]);
        (smem + N)[si[e]] = (u64)__double_as_longlong(a1[e]);
      }
    }
  }
  __syncthreads();
  mbar_wait(twbar, 1);
  {
    constexpr int R0 = ((LOGN - 1) % 3) + 1;
    const TwShared iw{TWb, qinv};
    auto pass_both = [&](auto s0, auto r) {
      constexpr int S0 = decltype(s0)::value, R = decltype(r)::value;
      f64_inv_pass<LOGN, NT, S0, R>(reinterpret_cast<double*>(smem), iw, qd, tid);
      f64_inv_pass<LOGN, NT, S0, R>(reinterpret_cast<double*>(smem + N), iw, qd, tid);
      __syncthreads();
    };
    if constexpr (LOGN > R0 + 9) pass_both(std::integral_constant<int, R0 + 9>{}, std::integral_constant<int, 3>{});
    if constexpr (LOGN > R0 + 6) pass_both(std::integral_constant<int, R0 + 6>{}, std::integral_constant<int, 3>{});
    if constexpr (LOGN > R0 + 3) pass_both(std::integral_constant<int, R0 + 3>{}, std::integral_constant<int, 3>{});
    if constexpr (LOGN > R0) pass_both(std::integral_constant<int, R0>{}, std::integral_constant<int, 3>{});
    pass_both(std::integral_constant<int, 0>{}, std::integral_constant<int, R0>{});
  }
  // ---- phase 3: final scaling; the special-prime CTA publishes its two accumulators through L2 ----
  if (I == k) {
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      u64* xo = L.xch + ((u64)z * 2 + c) * N;
      const u64* A = smem + (size_t)c * N;
#pragma unroll
      for (int i = tid; i < N; i += NT) xo[i] = eng_finish_inv_native<ENG_FP64>(A[swz(i)], i, mI);
    }
  } else {
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      u64* A = smem + (size_t)c * N;
      // N^-1 psi^-i scaling; the signed representative (|t| <= 0.54 q) is all the mod-down below needs
#pragma unroll
      for (int i = tid; i < N; i += NT) {
        const double2 f2 = __ldg(mI.fin + i);
        A[swz(i)] = (u64)__double_as_longlong(f64_modmul(__longlong_as_double((long long)A[swz(i)]), f2.x, f2.y, qd));
      }
    }
    // stage c0's polynomial of this modulus in the free table buffer: the Galois gather of phase 4 becomes a
    // shared-memory permutation
    const u64* sp = src + (u64)I * N;
    u64* SB = reinterpret_cast<u64*>(TWb);
#pragma unroll
    for (int i = tid; i < N; i += NT) SB[i] = sp[i];
  }
  cluster.sync();
  // ---- phase 4: mod-down by P of both components, add sigma_g(c0), expansion butterfly ----
  if (I < k) {
    const int j = I;
    const u64 q = mI.q;
    const u64* SB = reinterpret_cast<const u64*>(TWb);
    u64* dstE = work + qi * L.q_stride + L.dst_off[ti] + kk * ctL;
    const u32 s1 = (2 * N - (1u << L.j)) & (2 * N - 1);
    const double Pqd = P.m[k].qd;
    constexpr int CH = 4;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const u64* lastA = L.xch + ((u64)z * 2 + c) * N;
      const u64* A = smem + (size_t)c * N;
      const u64* sp1 = src + (u64)(k + j) * N;  // c1's polynomial of this modulus (coalesced reads)
#pragma unroll 1
      for (int i0 = tid; i0 < N; i0 += CH * NT) {
        u64 la[CH], av[CH], pv[CH], gv[CH];
#pragma unroll
        for (int e = 0; e < CH; ++e) {
          const int i = i0 + e * NT;
          la[e] = __ldcg(lastA + i);
          av[e] = A[swz(i)];
          gv[e] = (c == 0) ? galois_gather(SB, i, L.ginv, N, q) : 0;
          pv[e] = (mode == 1) ? 0 : (c == 0 ? SB[i] : sp1[i]);
        }
        // Everything stays an integer-valued double until the two outputs are canonicalised.  With l = (acc_P + P/2)
        // mod P in [0, P):  md = (a - l + (P/2 mod q)) * P^-1 mod q  — any representative of l mod q serves, since the
        // exact product only needs |y| < 2^48 — then E = p + (sigma_g(c0) +) md and O = +-(p - (sigma_g(c0) +) md).
#pragma unroll
        for (int e = 0; e < CH; ++e) {
          const int i = i0 + e * NT;
          double l = __dadd_rn(__longlong_as_double((long long)la[e]), P.half_P_d);
          l = l >= Pqd ? __dadd_rn(l, -Pqd) : l;
          const double dd = __dadd_rn(__dadd_rn(__longlong_as_double((long long)av[e]), -l), P.half_P_mod_d[j]);
          double md = f64_modmul(dd, P.inv_P_d[j], P.inv_P_di[j], qd);
          if (c == 0) md = __dadd_rn(md, u64_to_f64_exact(gv[e]));
          if (mode == 1) {
            dstE[(u64)(c * k + j) * N + i] = f64_to_u64_exact(f64_canon(md, qd, qinv));
          } else {
            const double pd = u64_to_f64_exact(pv[e]);
            dstE[(u64)(c * k + j) * N + i] = f64_to_u64_exact(f64_canon(__dadd_rn(pd, md), qd, qinv));
            const u32 rr = i + s1;
            double d = __dadd_rn(pd, -md);
            if (rr & N) d = -d;
            (dstE + ((u64)ctL << L.j))[(u64)(c * k + j) * N + (rr & (N - 1))] = f64_to_u64_exact(f64_canon(d, qd, qinv));
          }
        }
      }
    }
  }
}

static size_t ks_cluster_smem(int k, int logn, int engine) {
  const bool tws = engine == ENG_FP64 && logn <= 12;  // + staged twiddle table and its mbarrier
  return (size_t)((k + 1) / 2 + 1 + (tws ? 1 : 0)) * ((size_t)1 << logn) * sizeof(u64) + (tws ? 16 : 0);
}

static bool ks_cluster_fits(int k, int logn, int engine) {
  return 2 * (k + 1) <= 16 && ks_cluster_smem(k, logn, engine) <= 227 * 1024 && logn >= 11 && logn <= 14;
}

bool ks_cluster_supported(const DevParams& P) { return ks_cluster_fits(P.k, P.logn, P.ntt_engine); }

// the most dynamic shared memory any supported k needs at this N and engine (k selects no instantiation of its own)
static size_t ks_cluster_smem_max(int logn, int engine) {
  size_t most = 0;
  for (int k = 1; 2 * (k + 1) <= 16; ++k)
    if (ks_cluster_fits(k, logn, engine)) most = std::max(most, ks_cluster_smem(k, logn, engine));
  return most;
}

// second generation: FP64 engine, staged twiddles (N <= 4096), k <= 2 (k digit buffers + table fit twice per SM)
static bool ks_cluster2_supported(const DevParams& P) {
  return P.ntt_engine == ENG_FP64 && P.logn <= 12 && P.logn >= 11 && P.k <= 2;
}
template <int LN, int K>
static cudaError_t launch_cluster2(const DevParams& P, u64* work, const LevelArgs& L, const u64* key, int mode,
                                   unsigned nodes, cudaStream_t st) {
  auto kern = k_ks_level_cluster2<LN, K>;
  const size_t smem = (size_t)((K < 2 ? 2 : K) + 1) * P.N * sizeof(u64) + 16;
  static bool configured[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!configured[dev & 63]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    configured[dev & 63] = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(nodes * (K + 1));
  cfg.blockDim = dim3(CCfg<LN>::NT);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = K + 1;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  static const bool pdl = !(getenv("PIRB_PDL") && getenv("PIRB_PDL")[0] == '0');
  cfg.numAttrs = pdl ? 2 : 1;
  return cudaLaunchKernelEx(&cfg, kern, P, work, L, key, mode);
}

cudaError_t launch_ks_level_cluster(const DevParams& P, u64* work, const LevelArgs& L, const u64* key, int mode,
                                    cudaStream_t st) {
  const unsigned nodes = (unsigned)L.n_queries * L.n_trees << L.j;
  if (!nodes) return cudaSuccess;
  const int k = P.k;
  {
    // wide levels (enough nodes to fill every SM twice with the fatter CTAs) take the second generation; narrow levels
    // are latency-bound chains where the first generation's six short CTAs per node finish sooner
    static const int v2_min = getenv("PIRB_KS_V2_MIN_NODES") ? atoi(getenv("PIRB_KS_V2_MIN_NODES")) : 0;
    int sm = 148;
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, dev);
    const unsigned thresh = v2_min > 0 ? (unsigned)v2_min : (unsigned)(2 * sm / (k + 1));
    if (v2_min >= 0 && ks_cluster2_supported(P) && nodes >= thresh) {
      if (P.logn == 12 && k == 2) return launch_cluster2<12, 2>(P, work, L, key, mode, nodes, st);
      if (P.logn == 12 && k == 1) return launch_cluster2<12, 1>(P, work, L, key, mode, nodes, st);
      if (P.logn == 11 && k == 2) return launch_cluster2<11, 2>(P, work, L, key, mode, nodes, st);
      if (P.logn == 11 && k == 1) return launch_cluster2<11, 1>(P, work, L, key, mode, nodes, st);
    }
  }
  const unsigned csize = 2 * (k + 1);
  const size_t smem = ks_cluster_smem(k, P.logn, P.ntt_engine);
  auto go = [&](auto ln, auto lz, auto mm) -> cudaError_t {
    constexpr int LN = decltype(ln)::value;
    constexpr int LZ = decltype(lz)::value;
    constexpr int MM = decltype(mm)::value;
    auto kern = k_ks_level_cluster<LN, LZ, MM>;
    // Every k shares this instantiation, so it is configured once per device for the largest of them: the most shared
    // memory any k needs and clusters above the portable 8 CTAs (k >= 4).  A process may serve several parameter sets
    // in any order; k = 3 and k = 4 need the same bytes, and only the larger cluster needs the opt-in.
    static bool configured[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!configured[dev & 63]) {
      cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)ks_cluster_smem_max(LN, LZ));
      if (e != cudaSuccess) return e;
      e = cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
      if (e != cudaSuccess) return e;
      configured[dev & 63] = true;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(nodes * csize);
    cfg.blockDim = dim3(CCfg<LN>::NT);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = csize;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    static const bool pdl = !(getenv("PIRB_PDL") && getenv("PIRB_PDL")[0] == '0');
    cfg.numAttrs = pdl ? 2 : 1;
    return cudaLaunchKernelEx(&cfg, kern, P, work, L, key, mode);
  };
  auto by_mode = [&](auto ln, auto lz) -> cudaError_t {
    switch (P.mac_mode) {
      case MAC_FP64: return go(ln, lz, std::integral_constant<int, MAC_FP64>{});
      case MAC_INT24: return go(ln, lz, std::integral_constant<int, MAC_INT24>{});
      default: return go(ln, lz, std::integral_constant<int, MAC_WIDE>{});
    }
  };
#define PIRB_CASE(LN)                                                                             \
  case LN:                                                                                        \
    switch (P.ntt_engine) {                                                                       \
      case ENG_FP64: return by_mode(std::integral_constant<int, LN>{}, std::integral_constant<int, ENG_FP64>{});         \
      case ENG_INT_LAZY: return by_mode(std::integral_constant<int, LN>{}, std::integral_constant<int, ENG_INT_LAZY>{}); \
      default: return by_mode(std::integral_constant<int, LN>{}, std::integral_constant<int, ENG_INT>{});                \
    }
  switch (P.logn) {
    PIRB_CASE(11)
    PIRB_CASE(12)
    PIRB_CASE(13)
    PIRB_CASE(14)
    default: return cudaErrorInvalidValue;
  }
#undef PIRB_CASE
}

}  // namespace pirb
