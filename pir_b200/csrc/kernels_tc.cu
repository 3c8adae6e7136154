// kernels_tc.cu — the BATCHED database scan on the 5th-generation tensor cores (tcgen05.mma kind::i8, TMEM
// accumulators, TMA-fed shared-memory operands).
//
// Reference: DatabaseMultiplier::multiply, last dimension (database.cpp:185-194, 238-247): for every row r of the
// hypercube and every query q,  row[q][r] = sum_i1  sv[q][i1] (.) db[r*dimL + i1]   (NTT form, per coefficient, mod q_j).
// For ONE query that is a bandwidth-bound stream (k_scan).  For a batch of queries sharing one pass over the database
// (BASELINE configs[3]) it is, for every coefficient slot c, a dense integer contraction
//        [rows x dimL] x [dimL x 2Q]      (2 ciphertext polynomials per query)
// of residues below 2^(8*NB) (NB = 5 bytes for the 36-bit primes of N=4096, 6 for the 43/44-bit primes of N=8192).
// Residues are split into NB byte limbs and the contraction runs on the tensor cores as u8 x u8 -> s32:
//        D[(a, r)][(q, p, b)] = sum_i1  dbbyte_a[r][i1] * svbyte_b[q][p][i1]            (< 2^16 * dimL, exact in s32)
//        row[q][r][p] = ( sum_{a,b} D[(a,r)][(q,p,b)] * 2^(8(a+b)) ) mod q_j             (epilogue, exact)
// so the result is bit-identical to the integer path.  The database is kept in a second, byte-planar layout
//        dbT[c][tile][lane = a*RPT + r'][Kp]     u8, K-major, RPT = 128 / NB rows per 128-lane tile, Kp = dimL up to x16
// (5/8 or 6/8 of the bytes of the u64 layout) and the selection vectors of a call are repacked into
//        svT[c][n = (q*2 + p)*NB + b][Kp]        u8, K-major.
// One persistent CTA per SM walks over coefficient slots; per slot and query tile it keeps the B operand (all of K)
// resident in shared memory and streams the A tiles through a TMA ring:
//   warp 0     TMA producer (cp.async.bulk.tensor, 128B swizzle, mbarrier transaction counts)
//   warp 1     MMA issuer: one thread, tcgen05.mma.cta_group::1.kind::i8, M = 128, N = 16*NB*(QT/8), K = 32 per
//              instruction; tcgen05.commit releases ring stages / publishes accumulators
//   warp 2     TMEM allocation
//   warps 4-7 / 8-11   two epilogue groups, one per TMEM accumulator buffer: tcgen05.ld -> limb recombination ->
//              cross-lane (a) reduction through shared memory -> Barrett -> global
#include <cuda.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "kernels.cuh"
#include "pirb_device.cuh"

namespace pirb {

// ---------------------------------------------------------------------------------------------------------------
// PTX wrappers (sm_100a)
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, u64* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"((u64)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc(u32* dst_smem, u32 ncols) {  // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(u32 taddr, u32 ncols) {  // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_i8(u32 tmem_d, u64 adesc, u64 bdesc, u32 idesc, u32 accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(u64* bar) {  // arrives on bar when all MMAs issued so far have completed
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld16(u32 taddr, u32 (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// bounded mbarrier wait: a protocol bug must not hang the GPU.  Returns false after ~2 s and raises *err.
__device__ __forceinline__ bool mbar_wait_b(u64* bar, u32 parity, volatile int* err) {
  const u32 a = smem_u32(bar);
  for (u32 it = 0;; ++it) {
    u32 done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(a), "r"(parity)
        : "memory");
    if (done) return true;
    if (it > (1u << 22)) {  // each failed try_wait suspends for up to ~1 us of hardware time
      *err = 1;
      return false;
    }
    if ((it & 1023) == 1023 && *err) return false;
  }
}

// K-major, 128-byte-swizzled operand tile in shared memory (rows of 128 B, 8-row swizzle atoms of 1024 B):
// start address >> 4 in bits [0,14), stride between 8-row groups (1024 B) >> 4 in bits [32,46), descriptor version 1 in
// bits [46,48), layout type SWIZZLE_128B (= 2) in bits [61,64).  The leading-dimension offset is unused in this mode.
__device__ __forceinline__ u64 umma_desc_sw128(u32 smem_addr) {
  return (u64)((smem_addr & 0x3FFFFu) >> 4) | ((u64)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}

// ---------------------------------------------------------------------------------------------------------------
// layout conversions
// ---------------------------------------------------------------------------------------------------------------
// database u64 [pt][k][N] -> dbT (see header).  grid (tile, c / 32), block (32, 32); dbT must be zero-filled before.
__global__ void __launch_bounds__(1024)
k_tc_pack_db(const u64* __restrict__ db, u64 num_pt, u32 dimL, u32 n_rows, u32 kN, u32 nb, u32 rpt, u32 ntiles, u32 Kp,
             u8* __restrict__ dbT) {
  __shared__ u64 t[32][33];
  const u32 tile = blockIdx.x, c0 = blockIdx.y * 32;
  const u32 tx = threadIdx.x, ty = threadIdx.y;
  for (u32 rr = 0; rr < rpt; ++rr) {
    const u32 row = tile * rpt + rr;
    if (row >= n_rows) break;
    for (u32 i0 = 0; i0 < dimL; i0 += 32) {
      const u32 i = i0 + ty;
      const u64 pt = (u64)row * dimL + i;
      t[ty][tx] = (i < dimL && pt < num_pt) ? db[pt * kN + c0 + tx] : 0ull;
      __syncthreads();
      // thread (tx = i1 offset, ty = coefficient offset)
      const u64 v = t[tx][ty];
      if (i0 + tx < dimL) {
        u8* o = dbT + (((u64)(c0 + ty) * ntiles + tile) * 128 + rr) * Kp + i0 + tx;
        for (u32 a = 0; a < nb; ++a) o[(u64)a * rpt * Kp] = (u8)(v >> (8 * a));
      }
      __syncthreads();
    }
  }
}

// selection vectors u64 [q][i1][2][k][N] (NTT form, sv_qstride limbs between queries) -> rows [row0 + qp*nb, ...) of an
// svT array with n_rows_total rows per coefficient (see header).
// A block transposes a tile of 128 selection entries (one K chunk) x 64 coefficients through shared memory: every
// row of the tile is read as 512 contiguous bytes (all loads of a thread in flight before the first shared-memory
// store) and every (coefficient, limb byte) row of svT is written as the 128 contiguous bytes of the chunk.
// grid (q * 2 + p, c / 64, K chunk), block 512, 128 * 66 * 8 bytes of dynamic shared memory; the K padding of svT
// beyond Kp's last chunk stays zero from allocation.
constexpr int PACK_C = 64, PACK_PITCH = PACK_C + 2;
__global__ void __launch_bounds__(512, 2)
k_tc_pack_sv(const u64* __restrict__ sv, u64 sv_qstride, u32 dimL, u32 kN, u32 nb, u32 n_rows_total, u32 row0, u32 Kp,
             u8* __restrict__ svT) {
  extern __shared__ __align__(16) u64 t[];  // [128][PACK_PITCH]
  const u32 qp = blockIdx.x, c0 = blockIdx.y * PACK_C, i0 = blockIdx.z * 128;
  const u32 q = qp >> 1, p = qp & 1;
  const u32 lane = threadIdx.x & 31, w = threadIdx.x >> 5;  // 16 warps; a warp reads one row: 32 lanes x 2 coefficients
  ulonglong2 v[8];
#pragma unroll
  for (int x = 0; x < 8; ++x) {
    const u32 i = i0 + w + 16 * x;
    v[x] = make_ulonglong2(0, 0);
    if (i < dimL)
      v[x] = __ldg(reinterpret_cast<const ulonglong2*>(sv + (u64)q * sv_qstride + (u64)i * 2 * kN + (u64)p * kN + c0) + lane);
  }
#pragma unroll
  for (int x = 0; x < 8; ++x) *reinterpret_cast<ulonglong2*>(t + (size_t)(w + 16 * x) * PACK_PITCH + 2 * lane) = v[x];
  __syncthreads();
  // thread (coefficient cc, group g of 16 consecutive selection entries)
  const u32 cc = threadIdx.x & (PACK_C - 1), g = threadIdx.x / PACK_C;  // 8 groups
  const u32 ib = i0 + g * 16;
  if (ib < Kp) {
    u64 r64[16];
#pragma unroll
    for (int x = 0; x < 16; ++x) r64[x] = t[(size_t)(g * 16 + x) * PACK_PITCH + cc];
    u8* o = svT + ((u64)(c0 + cc) * n_rows_total + row0 + (u64)qp * nb) * Kp + ib;
    for (u32 b = 0; b < nb; ++b) {
      u32 r[4];
#pragma unroll
      for (int g4 = 0; g4 < 4; ++g4)
        r[g4] = (u32)((r64[g4 * 4] >> (8 * b)) & 0xFF) | ((u32)((r64[g4 * 4 + 1] >> (8 * b)) & 0xFF) << 8) |
                ((u32)((r64[g4 * 4 + 2] >> (8 * b)) & 0xFF) << 16) | ((u32)((r64[g4 * 4 + 3] >> (8 * b)) & 0xFF) << 24);
      *reinterpret_cast<uint4*>(o + (u64)b * Kp) = make_uint4(r[0], r[1], r[2], r[3]);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// the scan
// ---------------------------------------------------------------------------------------------------------------
struct TcScanArgs {
  u32 kN, n_rows, ntiles, rpt, Kp, kch;  // kch = K chunks of 128 bytes
  u32 n_queries;                          // real queries (outputs of padded ones are dropped)
  u32 n_qt, qt;                           // query tiles per coefficient, queries per tile (multiple of 8)
  u32 n_cols;                             // N of the MMA = qt * 2 * NB
  u32 sv_rows_total;                      // rows of svT per coefficient
  u32 sv_row0;                            // first row of this call's queries inside a coefficient's rows
  u32 stages, b_bufs;                     // A ring depth, B buffers (1 or 2)
  u32 n_acc;                              // TMEM accumulator buffers = epilogue groups (2..4)
  u64* part;                              // [q][row][2][k][N]
  int* err;
};

constexpr int TC_THREADS = 128 + 128 * TC_MAX_ACC;       // 4 control warps + 4 warps per epilogue group (tc_plan.h)

template <int NB>
__global__ void __launch_bounds__(TC_THREADS, 1)
k_tc_scan(const __grid_constant__ DevParams P, const __grid_constant__ CUtensorMap mapA,
          const __grid_constant__ CUtensorMap mapB, const TcScanArgs A) {
  extern __shared__ __align__(1024) u8 smem[];
  constexpr u32 EW = NB <= 5 ? 1 : 2;  // u64 words per recombined partial
  const u32 warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const u32 b_chunk_bytes = A.n_cols * 128;
  const u32 b_buf_bytes = A.kch * b_chunk_bytes;
  u8* sA = smem;
  u8* sB = sA + (size_t)A.stages * TC_A_STAGE_BYTES;
  u64* sE = reinterpret_cast<u64*>(sB + (size_t)A.b_bufs * b_buf_bytes);  // [2 groups][16 qp][128 lanes][EW]
  u64* bars = sE + (size_t)TC_MAX_ACC * 16 * 128 * EW;
  u64* a_full = bars;
  u64* a_empty = a_full + A.stages;
  u64* b_full = a_empty + A.stages;
  u64* b_empty = b_full + 2;
  u64* t_full = b_empty + 2;
  u64* t_empty = t_full + TC_MAX_ACC;
  u32* tmem_slot = reinterpret_cast<u32*>(t_empty + TC_MAX_ACC);
  volatile int* err = A.err;

  if (threadIdx.x == 0) {
    for (u32 s = 0; s < A.stages; ++s) { mbar_init(a_full + s, 1); mbar_init(a_empty + s, 1); }
    for (u32 s = 0; s < 2; ++s) {
      mbar_init(b_full + s, 1);
      mbar_init(b_empty + s, 1);
    }
    for (u32 s = 0; s < TC_MAX_ACC; ++s) {
      mbar_init(t_full + s, 1);
      mbar_init(t_empty + s, 4);  // one arrival per epilogue warp of the group
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  const u32 acc_stride = A.n_acc * A.n_cols <= 256 ? 256 / A.n_acc : 512 / A.n_acc;  // columns per accumulator buffer
  const u32 tmem_cols = A.n_acc * acc_stride;  // 256 or 512 for n_acc in {2, 4}
  if (warp == 2) tmem_alloc(tmem_slot, tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const u32 tmem_base = *tmem_slot;

  const u32 n_items = A.kN;
  if (warp == 0) {
    // ------------------------------------------------ TMA producer ------------------------------------------------
    if (lane == 0) {
      u32 st = 0, ph = 0, bcount = 0;
      bool ok = true;
      for (u32 c = blockIdx.x; c < n_items && ok; c += gridDim.x) {
        for (u32 qt = 0; qt < A.n_qt && ok; ++qt) {
          const u32 bb = A.b_bufs == 2 ? (bcount & 1) : 0;
          const u32 bph = A.b_bufs == 2 ? ((bcount >> 1) & 1) : (bcount & 1);
          ok = mbar_wait_b(b_empty + bb, bph ^ 1, err);
          if (!ok) break;
          mbar_expect_tx(b_full + bb, b_buf_bytes);
          for (u32 kc = 0; kc < A.kch; ++kc)
            tma_load_2d(sB + (size_t)bb * b_buf_bytes + (size_t)kc * b_chunk_bytes, &mapB, (int)(kc * 128),
                        (int)(c * A.sv_rows_total + A.sv_row0 + qt * A.n_cols), b_full + bb);
          ++bcount;
          for (u32 mt = 0; mt < A.ntiles && ok; ++mt)
            for (u32 kc = 0; kc < A.kch; ++kc) {
              ok = mbar_wait_b(a_empty + st, ph ^ 1, err);
              if (!ok) break;
              mbar_expect_tx(a_full + st, TC_A_STAGE_BYTES);
              tma_load_2d(sA + (size_t)st * TC_A_STAGE_BYTES, &mapA, (int)(kc * 128), (int)((c * A.ntiles + mt) * 128),
                          a_full + st);
              if (++st == A.stages) { st = 0; ph ^= 1; }
            }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------ MMA issuer --------------------------------------------------
    if (lane == 0) {
      // instruction descriptor: D = s32 (2 << 4), A and B unsigned 8-bit (0), both K-major, N >> 3 at bit 17, M >> 4 at 24
      const u32 idesc = (2u << 4) | ((A.n_cols >> 3) << 17) | ((128u >> 4) << 24);
      u32 st = 0, ph = 0, bcount = 0, tcount = 0;
      bool ok = true;
      for (u32 c = blockIdx.x; c < n_items && ok; c += gridDim.x) {
        for (u32 qt = 0; qt < A.n_qt && ok; ++qt) {
          const u32 bb = A.b_bufs == 2 ? (bcount & 1) : 0;
          const u32 bph = A.b_bufs == 2 ? ((bcount >> 1) & 1) : (bcount & 1);
          ok = mbar_wait_b(b_full + bb, bph, err);
          if (!ok) break;
          const u32 sB_addr = smem_u32(sB + (size_t)bb * b_buf_bytes);
          for (u32 mt = 0; mt < A.ntiles && ok; ++mt) {
            const u32 ab = tcount % A.n_acc, tph = (tcount / A.n_acc) & 1;
            ok = mbar_wait_b(t_empty + ab, tph ^ 1, err);
            if (!ok) break;
            tc_fence_after();
            const u32 d_addr = tmem_base + ab * acc_stride;
            for (u32 kc = 0; kc < A.kch; ++kc) {
              ok = mbar_wait_b(a_full + st, ph, err);
              if (!ok) break;
              tc_fence_after();
              const u64 ad = umma_desc_sw128(smem_u32(sA + (size_t)st * TC_A_STAGE_BYTES));
              const u64 bd = umma_desc_sw128(sB_addr + kc * b_chunk_bytes);
              const u32 kbytes = min(128u, A.Kp - kc * 128);
              const u32 nk = (kbytes + 31) / 32;
              for (u32 k = 0; k < nk; ++k) umma_i8(d_addr, ad + 2 * k, bd + 2 * k, idesc, (kc | k) != 0);
              umma_commit(a_empty + st);  // the stage is free once these MMAs have read it
              if (++st == A.stages) { st = 0; ph ^= 1; }
            }
            umma_commit(t_full + ab);
            ++tcount;
          }
          umma_commit(b_empty + bb);
          ++bcount;
        }
      }
    }
  } else if (warp >= 4 && ((warp - 4) >> 2) < A.n_acc) {
    // ------------------------------------------------ epilogue ----------------------------------------------------
    const u32 g = (warp - 4) >> 2;           // group <-> accumulator buffer
    const u32 wq = warp & 3;                 // TMEM lane quarter this warp may read
    const u32 m = wq * 32 + lane;            // accumulator lane = a * rpt + r'
    const u32 gt = threadIdx.x - 128 - g * 128;  // thread index within the group, 0..127
    u64* E = sE + (size_t)g * 16 * 128 * EW;
    const u32 n_pieces = A.qt / 8;           // 16 (q,p) pairs = 16 * NB columns per piece
    u32 tcount = 0;
    bool ok = true;
    for (u32 c = blockIdx.x; c < n_items && ok; c += gridDim.x) {
      const ModC& mod = P.m[c / P.N];
      for (u32 qt = 0; qt < A.n_qt && ok; ++qt)
        for (u32 mt = 0; mt < A.ntiles && ok; ++mt, ++tcount) {
          if (tcount % A.n_acc != g) continue;
          const u32 tph = (tcount / A.n_acc) & 1;
          ok = mbar_wait_b(t_full + g, tph, err);
          if (!ok) break;
          tc_fence_after();
          const u32 t_addr = tmem_base + g * acc_stride + ((wq * 32) << 16);
          for (u32 pc = 0; pc < n_pieces; ++pc) {
            u32 v[NB][16];
#pragma unroll
            for (int x = 0; x < NB; ++x) tmem_ld16(t_addr + pc * 16 * NB + x * 16, v[x]);
            tmem_ld_wait();
            if (pc == n_pieces - 1) {  // accumulator fully read: hand the buffer back to the MMA issuer
              tc_fence_before();
              __syncwarp();
              if (lane == 0) mbar_arrive(t_empty + g);
            }
            // limb recombination over b: 16 (q,p) pairs, NB consecutive columns each
            const u32* vf = &v[0][0];
#pragma unroll
            for (int qp = 0; qp < 16; ++qp) {
              if constexpr (NB <= 5) {
                u64 s = 0;
#pragma unroll
                for (int b = 0; b < NB; ++b) s += (u64)vf[qp * NB + b] << (8 * b);
                E[qp * 128 + m] = s;
              } else {
                u64 lo = 0, hi = 0;
#pragma unroll
                for (int b = 0; b < 4; ++b) lo += (u64)vf[qp * NB + b] << (8 * b);
#pragma unroll
                for (int b = 4; b < NB; ++b) hi += (u64)vf[qp * NB + b] << (8 * (b - 4));
                E[(qp * 128 + m) * 2] = lo;
                E[(qp * 128 + m) * 2 + 1] = hi;
              }
            }
            asm volatile("bar.sync %0, 128;" ::"r"(1 + g) : "memory");
            // cross-lane reduction over a, Barrett, store: rpt rows x 16 pairs per piece
            const u32 n_out = A.rpt * 16;
            for (u32 o = gt; o < n_out; o += 128) {
              const u32 qp = o / A.rpt, rr = o % A.rpt;
              u64 lo = 0, hi = 0;
#pragma unroll
              for (int a = 0; a < NB; ++a) {
                const u32 idx = qp * 128 + a * A.rpt + rr;
                if constexpr (NB <= 5) {
                  const u64 s = E[idx];
                  const u64 add_lo = s << (8 * a), add_hi = a ? (s >> (64 - 8 * a)) : 0;
                  lo += add_lo;
                  hi += add_hi + (lo < add_lo);
                } else {
                  const u64 s0 = E[idx * 2], s1 = E[idx * 2 + 1];
                  u64 add_lo = s0 << (8 * a), add_hi = a ? (s0 >> (64 - 8 * a)) : 0;
                  lo += add_lo;
                  hi += add_hi + (lo < add_lo);
                  const int sh = 32 + 8 * a;  // s1 * 2^sh, sh <= 72
                  if (sh < 64) { add_lo = s1 << sh; add_hi = s1 >> (64 - sh); }
                  else { add_lo = 0; add_hi = s1 << (sh - 64); }
                  lo += add_lo;
                  hi += add_hi + (lo < add_lo);
                }
              }
              const u32 q = qt * A.qt + pc * 8 + (qp >> 1), p = qp & 1;
              const u32 row = mt * A.rpt + rr;
              if (q < A.n_queries && row < A.n_rows)
                A.part[(((u64)q * A.n_rows + row) * 2 + p) * A.kN + c] = barrett128(lo, hi, mod.q, mod.ratio_hi, mod.ratio_lo);
            }
            asm volatile("bar.sync %0, 128;" ::"r"(1 + g) : "memory");  // E is rewritten by the next piece / tile
          }
        }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, tmem_cols);
}

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// 2D u8 tensor [rows][Kp] (Kp contiguous), box {128 bytes of K, box_rows}, 128-byte swizzle, zero fill out of bounds
static bool make_map(CUtensorMap* map, const void* base, u64 rows, u32 Kp, u32 box_rows) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return false;
  const cuuint64_t dims[2] = {Kp, rows};
  const cuuint64_t strides[1] = {Kp};
  const cuuint32_t box[2] = {128, box_rows};
  const cuuint32_t estr[2] = {1, 1};
  return fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

void tc_geometry(const DevParams& P, u32 dimL, u32 n_rows, TcGeom* g) {
  int max_bits = 0;
  for (int j = 0; j < P.k; ++j) max_bits = std::max(max_bits, 64 - __builtin_clzll(P.m[j].q));
  g->nb = (u32)(max_bits + 7) / 8;
  g->rpt = 128 / g->nb;
  g->ntiles = (n_rows + g->rpt - 1) / g->rpt;
  g->Kp = (dimL + 15) / 16 * 16;
  g->kch = (g->Kp + 127) / 128;
  g->db_bytes = (u64)P.k * P.N * g->ntiles * 128 * g->Kp;
}

bool tc_launch_plan(const DevParams& P, u32 dimL, u32 n_queries, TcPlan* plan) {
  TcGeom g;
  tc_geometry(P, dimL, 1, &g);
  // the operand repacking works on 64-coefficient blocks; the tensor maps need the driver's encoder
  if ((P.N % 64) != 0 || encode_fn() == nullptr) return false;
  const char* want = std::getenv("PIRB_TC_QT");
  return tc_plan(g.nb, dimL, n_queries, want ? atoi(want) : 16, plan);
}

cudaError_t launch_tc_pack_db(const DevParams& P, const u64* db, u64 num_pt, u32 dimL, u32 n_rows, const TcGeom& g,
                              u8* dbT, cudaStream_t st) {
  cudaError_t e = cudaMemsetAsync(dbT, 0, g.db_bytes, st);
  if (e != cudaSuccess) return e;
  const u32 kN = (u32)P.k * P.N;
  k_tc_pack_db<<<dim3(g.ntiles, kN / 32), dim3(32, 32), 0, st>>>(db, num_pt, dimL, n_rows, kN, g.nb, g.rpt, g.ntiles, g.Kp,
                                                                  dbT);
  return cudaGetLastError();
}

u64 tc_sv_bytes(const DevParams& P, const TcGeom& g, const TcPlan& plan) {
  return (u64)P.k * P.N * plan.n_qt * plan.n_cols * g.Kp;
}

cudaError_t launch_tc_pack_sv(const DevParams& P, const TcGeom& g, const u64* sv, u64 sv_qstride, u32 dimL, u32 n_queries,
                              u8* svT, u32 rows_total, u32 row0, cudaStream_t st) {
  if (!n_queries) return cudaSuccess;
  const u32 kN = (u32)P.k * P.N;
  const dim3 pgrid(n_queries * 2, kN / PACK_C, g.kch);
  const size_t psmem = (size_t)128 * PACK_PITCH * sizeof(u64);
  static bool configured[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!configured[dev & 63]) {
    cudaError_t e1 = cudaFuncSetAttribute(k_tc_pack_sv, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)psmem);
    if (e1 != cudaSuccess) return e1;
    configured[dev & 63] = true;
  }
  k_tc_pack_sv<<<pgrid, 512, psmem, st>>>(sv, sv_qstride, dimL, kN, g.nb, rows_total, row0, g.Kp, svT);
  return cudaGetLastError();
}

cudaError_t launch_tc_scan(const DevParams& P, const TcGeom& g, const TcPlan& plan, const u8* dbT, u32 dimL, u32 n_rows,
                           const u64* sv, u64 sv_qstride, u32 n_queries, u8* svT, int* err_flag, int sm_count, u64* part,
                           cudaStream_t st) {
  const u32 kN = (u32)P.k * P.N;
  const u32 sv_rows_total = plan.n_qt * plan.n_cols;
  // rows of padded queries must be zero; real ones are rewritten entirely (the K padding is never written)
  const u64 real_rows = (u64)n_queries * 2 * g.nb;
  if (real_rows < sv_rows_total) {
    cudaError_t e = cudaMemset2DAsync(svT + real_rows * g.Kp, (size_t)sv_rows_total * g.Kp, 0,
                                      (size_t)(sv_rows_total - real_rows) * g.Kp, kN, st);
    if (e != cudaSuccess) return e;
  }
  cudaError_t e = launch_tc_pack_sv(P, g, sv, sv_qstride, dimL, n_queries, svT, sv_rows_total, 0, st);
  if (e != cudaSuccess) return e;
  return launch_tc_scan_packed(P, g, plan, dbT, n_rows, svT, sv_rows_total, 0, n_queries, err_flag, sm_count, part, st);
}

cudaError_t launch_tc_scan_packed(const DevParams& P, const TcGeom& g, const TcPlan& plan, const u8* dbT, u32 n_rows,
                                  const u8* svT, u32 sv_rows_total, u32 row0, u32 n_queries, int* err_flag, int sm_count,
                                  u64* part, cudaStream_t st) {
  const u32 kN = (u32)P.k * P.N;
  const u32 n_cols = plan.n_cols;
  if (plan.Kp != g.Kp || plan.kch != g.kch || n_cols != plan.qt * 2 * g.nb || plan.n_qt * plan.qt < n_queries)
    return cudaErrorInvalidValue;  // a plan made for another shape

  CUtensorMap mapA, mapB;
  if (!make_map(&mapA, dbT, (u64)kN * g.ntiles * 128, g.Kp, 128)) return cudaErrorInvalidValue;
  if (!make_map(&mapB, svT, (u64)kN * sv_rows_total, g.Kp, n_cols)) return cudaErrorInvalidValue;

  TcScanArgs A;
  A.kN = kN;
  A.n_rows = n_rows;
  A.ntiles = g.ntiles;
  A.rpt = g.rpt;
  A.Kp = g.Kp;
  A.kch = g.kch;
  A.n_queries = n_queries;
  A.n_qt = plan.n_qt;
  A.qt = plan.qt;
  A.n_cols = n_cols;
  A.sv_rows_total = sv_rows_total;
  A.sv_row0 = row0;
  A.part = part;
  A.err = err_flag;
  A.n_acc = (TC_MAX_ACC >= 4 && 4 * n_cols <= 512) ? 4 : 2;  // accumulator buffers must fit the 512 TMEM columns
  A.b_bufs = plan.b_bufs;
  A.stages = plan.stages;
  const size_t smem = plan.smem;
  const int grid = std::min<int>(sm_count, (int)kN);
  auto go = [&](auto kern) -> cudaError_t {
    cudaError_t e2 = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e2 != cudaSuccess) return e2;
    kern<<<grid, TC_THREADS, smem, st>>>(P, mapA, mapB, A);
    return cudaGetLastError();
  };
  return g.nb == 5 ? go(k_tc_scan<5>) : go(k_tc_scan<6>);
}

}  // namespace pirb
