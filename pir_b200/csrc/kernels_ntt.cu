// kernels_ntt.cu — every kernel built around the shared-memory NTT core:
//   k_ntt_fwd / k_ntt_inv     Evaluator::transform_to/from_ntt_inplace (database.cpp:190,222,252)
//   k_db_preprocess           PIRDatabase::populate's transform_to_ntt_inplace(pt, first_parms_id) (database.cpp:103-106)
//   k_ks_digits / k_ks_mac_intt   Evaluator::apply_galois_inplace -> switch_key_inplace (server.cpp:71; SURVEY A.5)
//   k_reencode_ntt            CiphertextReencoder::Encode + plaintext NTT (ct_reencoder.cpp:40-71, database.cpp:217-228)
// One CTA owns one size-N transform; the polynomial lives in (swizzled) shared memory between
// a fused load-side transform and a fused store-side transform.
#include <cstdlib>
#include <set>
#include <type_traits>
#include <utility>

#include "kernels.cuh"
#include "pirb_device.cuh"

namespace pirb {

template <int LOGN>
struct Cfg {
  static constexpr int N = 1 << LOGN;
  static constexpr int NT = (N / 8 < 512) ? N / 8 : 512;
  static constexpr size_t SMEM = sizeof(u64) * N;
  static constexpr int MINB = LOGN <= 13 ? 2 : 1;  // resident CTAs per SM the register budget must allow
};

// ---------------------------------------------------------------------------------------------
template <int LOGN, int ENG>
__global__ void __launch_bounds__(Cfg<LOGN>::NT, Cfg<LOGN>::MINB)
k_ntt_fwd(const __grid_constant__ DevParams P, const u64* __restrict__ in, u64* __restrict__ out, int cycle, int off,
          u64 in_bstride, u64 out_bstride) {
  constexpr int N = Cfg<LOGN>::N, NT = Cfg<LOGN>::NT;
  extern __shared__ u64 s[];
  const int tid = threadIdx.x;
  const int p = blockIdx.x;
  const ModC& m = P.m[(p % cycle) + off];
  const u64* src = in + blockIdx.y * in_bstride + (u64)p * N;
  u64* dst = out + blockIdx.y * out_bstride + (u64)p * N;
#pragma unroll
  for (int i = tid; i < N; i += NT) s[swz(i)] = eng_load<ENG>(src[i]);
  __syncthreads();
  eng_forward<LOGN, NT, ENG>(s, m, tid);
#pragma unroll
  for (int i = tid; i < N; i += NT) dst[i] = eng_store_fwd<ENG>(s[swz(i)], m);
}

template <int LOGN, int ENG>
__global__ void __launch_bounds__(Cfg<LOGN>::NT, Cfg<LOGN>::MINB)
k_ntt_inv(const __grid_constant__ DevParams P, const u64* __restrict__ in, u64* __restrict__ out, int cycle, int off,
          int n_parts, u64 part_stride, u64 in_bstride, u64 out_bstride) {
  constexpr int N = Cfg<LOGN>::N, NT = Cfg<LOGN>::NT;
  extern __shared__ u64 s[];
  const int tid = threadIdx.x;
  const int p = blockIdx.x;
  const ModC& m = P.m[(p % cycle) + off];
  const u64* src = in + blockIdx.y * in_bstride + (u64)p * N;
  u64* dst = out + blockIdx.y * out_bstride + (u64)p * N;
#pragma unroll
  for (int i = tid; i < N; i += NT) {
    u64 v = src[i];
    for (int g = 1; g < n_parts; ++g) v = addmod(v, src[g * part_stride + i], m.q);
    s[swz(i)] = eng_load<ENG>(v);
  }
  __syncthreads();
  eng_inverse<LOGN, NT, ENG>(s, m, tid);
#pragma unroll
  for (int i = tid; i < N; i += NT) dst[i] = eng_store_inv<ENG>(s[swz(i)], i, m);
}

// plaintext coefficient c (< t) -> c >= (t+1)/2 ? c + (q_j - t) : c   (SURVEY A.7), then NTT mod q_j
template <int LOGN, int ENG>
__global__ void __launch_bounds__(Cfg<LOGN>::NT, Cfg<LOGN>::MINB)
k_db_preprocess(const __grid_constant__ DevParams P, const u64* __restrict__ coeffs, u64* __restrict__ out) {
  constexpr int N = Cfg<LOGN>::N, NT = Cfg<LOGN>::NT;
  extern __shared__ u64 s[];
  const int tid = threadIdx.x;
  const int j = blockIdx.y;
  const u64 pt = blockIdx.x;
  const ModC& m = P.m[j];
  const u64* src = coeffs + pt * N;
  u64* dst = out + (pt * P.k + j) * N;
  const u64 inc = m.q - P.t;
#pragma unroll
  for (int i = tid; i < N; i += NT) {
    u64 c = src[i];
    s[swz(i)] = eng_load<ENG>(c >= P.thr ? c + inc : c);
  }
  __syncthreads();
  eng_forward<LOGN, NT, ENG>(s, m, tid);
#pragma unroll
  for (int i = tid; i < N; i += NT) dst[i] = eng_store_fwd<ENG>(s[swz(i)], m);
}

// grid (z = node, I = key-level modulus, J = RNS digit)
template <int LOGN, int ENG>
__global__ void __launch_bounds__(Cfg<LOGN>::NT, Cfg<LOGN>::MINB)
k_ks_digits(const __grid_constant__ DevParams P, const u64* __restrict__ work, const LevelArgs L,
            u64* __restrict__ dig) {
  constexpr int N = Cfg<LOGN>::N, NT = Cfg<LOGN>::NT;
  extern __shared__ u64 s[];
  const int tid = threadIdx.x;
  const int I = blockIdx.y, J = blockIdx.z;
  const u32 z = blockIdx.x;
  const u32 kk = z & ((1u << L.j) - 1);
  const u32 tq = z >> L.j;
  const u32 ti = tq % L.n_trees, qi = tq / L.n_trees;
  const int k = P.k;
  const u64 ctL = (u64)2 * k * N;
  const u64* c1 = work + qi * L.q_stride + L.src_off[ti] + kk * ctL + (u64)(k + J) * N;
  const ModC& mI = P.m[I];
  const u64 qJ = P.m[J].q;
  const bool need_reduce = qJ > mI.q;
#pragma unroll
  for (int i = tid; i < N; i += NT) {
    u64 v = galois_gather(c1, i, L.ginv, N, qJ);
    if (need_reduce) v = barrett64(v, mI.q, mI.ratio_hi);
    s[swz(i)] = eng_load<ENG>(v);
  }
  __syncthreads();
  eng_forward<LOGN, NT, ENG>(s, mI, tid);
  u64* dst = dig + (((u64)z * (k + 1) + I) * k + J) * N;
#pragma unroll
  for (int i = tid; i < N; i += NT) dst[i] = eng_store_fwd<ENG>(s[swz(i)], mI);
}

// grid (z = node, I, c = key component)
template <int LOGN, int ENG>
__global__ void __launch_bounds__(Cfg<LOGN>::NT, Cfg<LOGN>::MINB)
k_ks_mac_intt(const __grid_constant__ DevParams P, const u64* __restrict__ dig, const u64* __restrict__ key_arg,
              u64* __restrict__ acc, const u64* const* __restrict__ key_tab, u32 nodes_per_query) {
  constexpr int N = Cfg<LOGN>::N, NT = Cfg<LOGN>::NT;
  extern __shared__ u64 s[];
  const int tid = threadIdx.x;
  const int I = blockIdx.y, c = blockIdx.z;
  const u32 z = blockIdx.x;
  const u64* __restrict__ key = key_tab ? key_tab[z / nodes_per_query] : key_arg;
  const int k = P.k;
  const ModC& mI = P.m[I];
  const u64* d = dig + ((u64)z * (k + 1) + I) * k * N;
#pragma unroll
  for (int i = tid; i < N; i += NT) {
    u64 lo = 0, hi = 0;
    for (int J = 0; J < k; ++J) {
      const u64 kv = __ldg(key + ((u64)(J * 2 + c) * (k + 1) + I) * N + i);
      mac128(lo, hi, d[(u64)J * N + i], kv);
    }
    s[swz(i)] = eng_load<ENG>(barrett128(lo, hi, mI.q, mI.ratio_hi, mI.ratio_lo));
  }
  __syncthreads();
  eng_inverse<LOGN, NT, ENG>(s, mI, tid);
  u64* dst = acc + (((u64)z * 2 + c) * (k + 1) + I) * N;
#pragma unroll
  for (int i = tid; i < N; i += NT) dst[i] = eng_store_inv<ENG>(s[swz(i)], i, mI);
}

// grid (x = ciphertext, e = chunk, j' = target data modulus)
template <int LOGN, int ENG>
__global__ void __launch_bounds__(Cfg<LOGN>::NT, Cfg<LOGN>::MINB)
k_reencode_ntt(const __grid_constant__ DevParams P, const u64* __restrict__ cts, u64* __restrict__ pts) {
  constexpr int N = Cfg<LOGN>::N, NT = Cfg<LOGN>::NT;
  extern __shared__ u64 s[];
  const int tid = threadIdx.x;
  const int jp = blockIdx.z, e = blockIdx.y;
  const u64 x = blockIdx.x;
  const int k = P.k;
  const ModC& m = P.m[jp];
  const u64* src = cts + (x * 2 * k + (u64)P.re_poly[e] * k + P.re_mod[e]) * N;
  const u32 shift = P.re_shift[e];
  const u64 mask = (u64)((1u << P.ptb) - 1);
  const u64 inc = m.q - P.t;
#pragma unroll
  for (int i = tid; i < N; i += NT) {
    u64 c = (src[i] >> shift) & mask;
    s[swz(i)] = eng_load<ENG>(c >= P.thr ? c + inc : c);
  }
  __syncthreads();
  eng_forward<LOGN, NT, ENG>(s, m, tid);
  u64* dst = pts + ((x * P.two_er + e) * k + jp) * N;
#pragma unroll
  for (int i = tid; i < N; i += NT) dst[i] = eng_store_fwd<ENG>(s[swz(i)], m);
}

// ---------------------------------------------------------------------------------------------
// FP64 engine, N <= 4096: TWO polynomials of the same modulus per CTA.  The w-only twiddle table is staged in shared
// memory by one bulk asynchronous copy (the passes form w/q on the fly), both transforms run through the same passes
// and share every block barrier.  The one-polynomial kernels above fetched a (w, w/q) pair per twiddle through L1 and
// were bound by the load/store unit (~45 % of the FP64 pipe); these are used wherever polynomials pair up.
//   shared memory: [2][N] data + [N] table + mbarrier
// ---------------------------------------------------------------------------------------------
template <int LOGN>
struct Cfg2 {
  static constexpr int N = 1 << LOGN;
  static constexpr int NT = (N / 8 < 512) ? N / 8 : 512;
  static constexpr size_t SMEM = sizeof(u64) * N * 3 + 16;
};

template <int LOGN, bool INVERSE>
__device__ __forceinline__ void ntt2_stage_table(const ModC& m, double* TW, u64* bar, int tid) {
  if (tid == 0) {
    mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    mbar_expect_tx(bar, (1u << LOGN) * 8);
    bulk_g2s_plain(TW, INVERSE ? m.iw1 : m.fw1, (1u << LOGN) * 8, bar);
  }
}
template <int LOGN, int NT>
__device__ __forceinline__ void ntt2_forward(u64* s, const double* TW, const ModC& m, int tid) {
  constexpr int N = 1 << LOGN;
  constexpr int R0 = ((LOGN - 1) % 3) + 1;
  const TwShared tw{TW, m.qinv};
  double* a = reinterpret_cast<double*>(s);
  double* b = reinterpret_cast<double*>(s + N);
  f64_fwd_pass<LOGN, NT, 0, R0>(a, tw, m.qd, tid);
  f64_fwd_pass<LOGN, NT, 0, R0>(b, tw, m.qd, tid);
  __syncthreads();
  if constexpr (LOGN > R0) { f64_fwd_pass<LOGN, NT, R0, 3>(a, tw, m.qd, tid); f64_fwd_pass<LOGN, NT, R0, 3>(b, tw, m.qd, tid); __syncthreads(); }
  if constexpr (LOGN > R0 + 3) { f64_fwd_pass<LOGN, NT, R0 + 3, 3>(a, tw, m.qd, tid); f64_fwd_pass<LOGN, NT, R0 + 3, 3>(b, tw, m.qd, tid); __syncthreads(); }
  if constexpr (LOGN > R0 + 6) { f64_fwd_pass<LOGN, NT, R0 + 6, 3>(a, tw, m.qd, tid); f64_fwd_pass<LOGN, NT, R0 + 6, 3>(b, tw, m.qd, tid); __syncthreads(); }
  if constexpr (LOGN > R0 + 9) { f64_fwd_pass<LOGN, NT, R0 + 9, 3>(a, tw, m.qd, tid); f64_fwd_pass<LOGN, NT, R0 + 9, 3>(b, tw, m.qd, tid); __syncthreads(); }
}
template <int LOGN, int NT>
__device__ __forceinline__ void ntt2_inverse(u64* s, const double* TW, const ModC& m, int tid) {
  constexpr int N = 1 << LOGN;
  constexpr int R0 = ((LOGN - 1) % 3) + 1;
  const TwShared iw{TW, m.qinv};
  double* a = reinterpret_cast<double*>(s);
  double* b = reinterpret_cast<double*>(s + N);
  if constexpr (LOGN > R0 + 9) { f64_inv_pass<LOGN, NT, R0 + 9, 3>(a, iw, m.qd, tid); f64_inv_pass<LOGN, NT, R0 + 9, 3>(b, iw, m.qd, tid); __syncthreads(); }
  if constexpr (LOGN > R0 + 6) { f64_inv_pass<LOGN, NT, R0 + 6, 3>(a, iw, m.qd, tid); f64_inv_pass<LOGN, NT, R0 + 6, 3>(b, iw, m.qd, tid); __syncthreads(); }
  if constexpr (LOGN > R0 + 3) { f64_inv_pass<LOGN, NT, R0 + 3, 3>(a, iw, m.qd, tid); f64_inv_pass<LOGN, NT, R0 + 3, 3>(b, iw, m.qd, tid); __syncthreads(); }
  if constexpr (LOGN > R0) { f64_inv_pass<LOGN, NT, R0, 3>(a, iw, m.qd, tid); f64_inv_pass<LOGN, NT, R0, 3>(b, iw, m.qd, tid); __syncthreads(); }
  f64_inv_pass<LOGN, NT, 0, R0>(a, iw, m.qd, tid);
  f64_inv_pass<LOGN, NT, 0, R0>(b, iw, m.qd, tid);
  __syncthreads();
}

// polynomials p0 = (blockIdx.x / cycle) * 2 * cycle + blockIdx.x % cycle and p0 + cycle (same modulus)
template <int LOGN>
__global__ void __launch_bounds__(Cfg2<LOGN>::NT, 2)
k_ntt_fwd2(const __grid_constant__ DevParams P, const u64* __restrict__ in, u64* __restrict__ out, int cycle, int off,
           u64 in_bstride, u64 out_bstride) {
  constexpr int N = Cfg2<LOGN>::N, NT = Cfg2<LOGN>::NT;
  extern __shared__ u64 s[];
  const int tid = threadIdx.x;
  const int j = blockIdx.x % cycle;
  const u64 p0 = (u64)(blockIdx.x / cycle) * 2 * cycle + j;
  const ModC& m = P.m[j + off];
  double* TW = reinterpret_cast<double*>(s + 2 * N);
  u64* bar = s + 3 * N;
  ntt2_stage_table<LOGN, false>(m, TW, bar, tid);
  const u64* src = in + blockIdx.y * in_bstride + p0 * N;
  u64* dst = out + blockIdx.y * out_bstride + p0 * N;
#pragma unroll
  for (int i = tid; i < N; i += NT) {
    s[swz(i)] = eng_load<ENG_FP64>(src[i]);
    s[N + swz(i)] = eng_load<ENG_FP64>(src[(u64)cycle * N + i]);
  }
  __syncthreads();
  mbar_wait(bar, 0);
  ntt2_forward<LOGN, NT>(s, TW, m, tid);
#pragma unroll
  for (int i = tid; i < N; i += NT) {
    dst[i] = eng_store_fwd<ENG_FP64>(s[swz(i)], m);
    dst[(u64)cycle * N + i] = eng_store_fwd<ENG_FP64>(s[N + swz(i)], m);
  }
}

template <int LOGN>
__global__ void __launch_bounds__(Cfg2<LOGN>::NT, 2)
k_ntt_inv2(const __grid_constant__ DevParams P, const u64* __restrict__ in, u64* __restrict__ out, int cycle, int off,
           int n_parts, u64 part_stride, u64 in_bstride, u64 out_bstride) {
  constexpr int N = Cfg2<LOGN>::N, NT = Cfg2<LOGN>::NT;
  extern __shared__ u64 s[];
  const int tid = threadIdx.x;
  const int j = blockIdx.x % cycle;
  const u64 p0 = (u64)(blockIdx.x / cycle) * 2 * cycle + j;
  const ModC& m = P.m[j + off];
  double* TW = reinterpret_cast<double*>(s + 2 * N);
  u64* bar = s + 3 * N;
  ntt2_stage_table<LOGN, true>(m, TW, bar, tid);
  const u64* src = in + blockIdx.y * in_bstride + p0 * N;
  u64* dst = out + blockIdx.y * out_bstride + p0 * N;
#pragma unroll
  for (int i = tid; i < N; i += NT) {
    u64 v = src[i], w = src[(u64)cycle * N + i];
    for (int g = 1; g < n_parts; ++g) {
      v = addmod(v, src[g * part_stride + i], m.q);
      w = addmod(w, src[g * part_stride + (u64)cycle * N + i], m.q);
    }
    s[swz(i)] = eng_load<ENG_FP64>(v);
    s[N + swz(i)] = eng_load<ENG_FP64>(w);
  }
  __syncthreads();
  mbar_wait(bar, 0);
  ntt2_inverse<LOGN, NT>(s, TW, m, tid);
#pragma unroll
  for (int i = tid; i < N; i += NT) {
    dst[i] = eng_store_inv<ENG_FP64>(s[swz(i)], i, m);
    dst[(u64)cycle * N + i] = eng_store_inv<ENG_FP64>(s[N + swz(i)], i, m);
  }
}

// grid (x = ciphertext, e2 = pair of chunks (2*e2, 2*e2 + 1), j' = target data modulus)
template <int LOGN>
__global__ void __launch_bounds__(Cfg2<LOGN>::NT, 2)
k_reencode_ntt2(const __grid_constant__ DevParams P, const u64* __restrict__ cts, u64* __restrict__ pts) {
  constexpr int N = Cfg2<LOGN>::N, NT = Cfg2<LOGN>::NT;
  extern __shared__ u64 s[];
  const int tid = threadIdx.x;
  const int jp = blockIdx.z, e0 = blockIdx.y * 2;
  const u64 x = blockIdx.x;
  const int k = P.k;
  const ModC& m = P.m[jp];
  double* TW = reinterpret_cast<double*>(s + 2 * N);
  u64* bar = s + 3 * N;
  ntt2_stage_table<LOGN, false>(m, TW, bar, tid);
  const u64 mask = (u64)((1u << P.ptb) - 1);
  const u64 inc = m.q - P.t;
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int e = e0 + h;
    const u64* src = cts + (x * 2 * k + (u64)P.re_poly[e] * k + P.re_mod[e]) * N;
    const u32 shift = P.re_shift[e];
#pragma unroll
    for (int i = tid; i < N; i += NT) {
      const u64 c = (src[i] >> shift) & mask;
      s[h * N + swz(i)] = eng_load<ENG_FP64>(c >= P.thr ? c + inc : c);
    }
  }
  __syncthreads();
  mbar_wait(bar, 0);
  ntt2_forward<LOGN, NT>(s, TW, m, tid);
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    u64* dst = pts + ((x * P.two_er + e0 + h) * k + jp) * N;
#pragma unroll
    for (int i = tid; i < N; i += NT) dst[i] = eng_store_fwd<ENG_FP64>(s[h * N + swz(i)], m);
  }
}

static bool ntt2_ok(const DevParams& P) {
  static const bool off = getenv("PIRB_NTT2") && getenv("PIRB_NTT2")[0] == '0';
  return !off && P.ntt_engine == ENG_FP64 && P.logn <= 12 && P.logn >= 11;
}
template <typename K>
static cudaError_t ensure_smem2(K kernel, size_t bytes);

// ---------------------------------------------------------------------------------------------
// host-side dispatch on log2(N) and on the NTT engine
// ---------------------------------------------------------------------------------------------
template <typename K>
static cudaError_t ensure_smem(K kernel, size_t bytes) {
  if (bytes <= 48 * 1024) return cudaSuccess;
  static std::set<std::pair<int, const void*>> configured;  // (device, kernel) pairs already set up
  int dev = 0;
  cudaGetDevice(&dev);
  const auto key = std::make_pair(dev, reinterpret_cast<const void*>(kernel));
  if (configured.count(key)) return cudaSuccess;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e == cudaSuccess) configured.insert(key);
  return e;
}

template <typename K>
static cudaError_t ensure_smem2(K kernel, size_t bytes) { return ensure_smem(kernel, bytes); }

template <int V>
using IntC = std::integral_constant<int, V>;

template <typename F>
static cudaError_t dispatch(const DevParams& P, F&& f) {
#define PIRB_CASE(LN)                                                   \
  case LN:                                                              \
    switch (P.ntt_engine) {                                             \
      case ENG_FP64: return f(IntC<LN>{}, IntC<ENG_FP64>{});            \
      case ENG_INT_LAZY: return f(IntC<LN>{}, IntC<ENG_INT_LAZY>{});    \
      default: return f(IntC<LN>{}, IntC<ENG_INT>{});                   \
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

cudaError_t launch_ntt_fwd(const DevParams& P, const u64* in, u64* out, int n_polys, int cycle, int off, int n_batch,
                           u64 in_bstride, u64 out_bstride, cudaStream_t st) {
  if (n_polys <= 0 || n_batch <= 0) return cudaSuccess;
  if (ntt2_ok(P) && n_polys % (2 * cycle) == 0) {  // polynomials p and p + cycle share a modulus: two per CTA
    auto go2 = [&](auto ln) -> cudaError_t {
      constexpr int LN = decltype(ln)::value;
      auto kern = k_ntt_fwd2<LN>;
      cudaError_t e = ensure_smem2(kern, Cfg2<LN>::SMEM);
      if (e != cudaSuccess) return e;
      kern<<<dim3(n_polys / 2, n_batch), Cfg2<LN>::NT, Cfg2<LN>::SMEM, st>>>(P, in, out, cycle, off, in_bstride, out_bstride);
      return cudaGetLastError();
    };
    return P.logn == 12 ? go2(IntC<12>{}) : go2(IntC<11>{});
  }
  return dispatch(P, [&](auto ln, auto lz) {
    constexpr int LN = decltype(ln)::value;
    constexpr int LZ = decltype(lz)::value;
    auto kern = k_ntt_fwd<LN, LZ>;
    cudaError_t e = ensure_smem(kern, Cfg<LN>::SMEM);
    if (e != cudaSuccess) return e;
    kern<<<dim3(n_polys, n_batch), Cfg<LN>::NT, Cfg<LN>::SMEM, st>>>(P, in, out, cycle, off, in_bstride, out_bstride);
    return cudaGetLastError();
  });
}

cudaError_t launch_ntt_inv(const DevParams& P, const u64* in, u64* out, int n_polys, int cycle, int off, int n_parts,
                           u64 part_stride, int n_batch, u64 in_bstride, u64 out_bstride, cudaStream_t st) {
  if (n_polys <= 0 || n_batch <= 0) return cudaSuccess;
  if (ntt2_ok(P) && n_polys % (2 * cycle) == 0) {
    auto go2 = [&](auto ln) -> cudaError_t {
      constexpr int LN = decltype(ln)::value;
      auto kern = k_ntt_inv2<LN>;
      cudaError_t e = ensure_smem2(kern, Cfg2<LN>::SMEM);
      if (e != cudaSuccess) return e;
      kern<<<dim3(n_polys / 2, n_batch), Cfg2<LN>::NT, Cfg2<LN>::SMEM, st>>>(P, in, out, cycle, off, n_parts, part_stride,
                                                                            in_bstride, out_bstride);
      return cudaGetLastError();
    };
    return P.logn == 12 ? go2(IntC<12>{}) : go2(IntC<11>{});
  }
  return dispatch(P, [&](auto ln, auto lz) {
    constexpr int LN = decltype(ln)::value;
    constexpr int LZ = decltype(lz)::value;
    auto kern = k_ntt_inv<LN, LZ>;
    cudaError_t e = ensure_smem(kern, Cfg<LN>::SMEM);
    if (e != cudaSuccess) return e;
    kern<<<dim3(n_polys, n_batch), Cfg<LN>::NT, Cfg<LN>::SMEM, st>>>(P, in, out, cycle, off, n_parts, part_stride,
                                                                     in_bstride, out_bstride);
    return cudaGetLastError();
  });
}

cudaError_t launch_db_preprocess(const DevParams& P, const u64* coeffs, u64* out, u64 n_pt, cudaStream_t st) {
  if (!n_pt) return cudaSuccess;
  return dispatch(P, [&](auto ln, auto lz) {
    constexpr int LN = decltype(ln)::value;
    constexpr int LZ = decltype(lz)::value;
    auto kern = k_db_preprocess<LN, LZ>;
    cudaError_t e = ensure_smem(kern, Cfg<LN>::SMEM);
    if (e != cudaSuccess) return e;
    kern<<<dim3((unsigned)n_pt, P.k), Cfg<LN>::NT, Cfg<LN>::SMEM, st>>>(P, coeffs, out);
    return cudaGetLastError();
  });
}

cudaError_t launch_ks_digits(const DevParams& P, const u64* work, const LevelArgs& L, u64* dig, cudaStream_t st) {
  const unsigned nodes = (unsigned)L.n_queries * L.n_trees << L.j;
  if (!nodes) return cudaSuccess;
  return dispatch(P, [&](auto ln, auto lz) {
    constexpr int LN = decltype(ln)::value;
    constexpr int LZ = decltype(lz)::value;
    auto kern = k_ks_digits<LN, LZ>;
    cudaError_t e = ensure_smem(kern, Cfg<LN>::SMEM);
    if (e != cudaSuccess) return e;
    kern<<<dim3(nodes, P.k + 1, P.k), Cfg<LN>::NT, Cfg<LN>::SMEM, st>>>(P, work, L, dig);
    return cudaGetLastError();
  });
}

cudaError_t launch_ks_mac_intt(const DevParams& P, const u64* dig, const u64* key, u64* acc, int n_nodes,
                               cudaStream_t st, const u64* const* key_tab, u32 nodes_per_query) {
  if (n_nodes <= 0) return cudaSuccess;
  return dispatch(P, [&](auto ln, auto lz) {
    constexpr int LN = decltype(ln)::value;
    constexpr int LZ = decltype(lz)::value;
    auto kern = k_ks_mac_intt<LN, LZ>;
    cudaError_t e = ensure_smem(kern, Cfg<LN>::SMEM);
    if (e != cudaSuccess) return e;
    kern<<<dim3(n_nodes, P.k + 1, 2), Cfg<LN>::NT, Cfg<LN>::SMEM, st>>>(P, dig, key, acc, key_tab, nodes_per_query);
    return cudaGetLastError();
  });
}

cudaError_t launch_reencode_ntt(const DevParams& P, const u64* cts, u64* pts, int n_cts, cudaStream_t st) {
  if (n_cts <= 0) return cudaSuccess;
  if (ntt2_ok(P) && P.two_er % 2 == 0) {  // chunks 2e and 2e + 1 go to the same target modulus: two per CTA
    auto go2 = [&](auto ln) -> cudaError_t {
      constexpr int LN = decltype(ln)::value;
      auto kern = k_reencode_ntt2<LN>;
      cudaError_t e = ensure_smem2(kern, Cfg2<LN>::SMEM);
      if (e != cudaSuccess) return e;
      kern<<<dim3(n_cts, P.two_er / 2, P.k), Cfg2<LN>::NT, Cfg2<LN>::SMEM, st>>>(P, cts, pts);
      return cudaGetLastError();
    };
    return P.logn == 12 ? go2(IntC<12>{}) : go2(IntC<11>{});
  }
  return dispatch(P, [&](auto ln, auto lz) {
    constexpr int LN = decltype(ln)::value;
    constexpr int LZ = decltype(lz)::value;
    auto kern = k_reencode_ntt<LN, LZ>;
    cudaError_t e = ensure_smem(kern, Cfg<LN>::SMEM);
    if (e != cudaSuccess) return e;
    kern<<<dim3(n_cts, P.two_er, P.k), Cfg<LN>::NT, Cfg<LN>::SMEM, st>>>(P, cts, pts);
    return cudaGetLastError();
  });
}

}  // namespace pirb
