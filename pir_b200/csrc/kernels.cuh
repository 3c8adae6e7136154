// kernels.cuh — launch wrappers of the sm_100a kernels of the PIR answer path (implemented in kernels_*.cu).
#pragma once
#include <cuda_runtime.h>

#include "pirb_common.h"
#include "tc_plan.h"

namespace pirb {

// One expansion level over a batch of trees (SURVEY §3.1 HOT LOOP 1).  Node z of the launch maps to
// (query qi, tree ti, node kk) with z = (qi * n_trees + ti) << j | kk; its source ciphertext is
// work + qi*q_stride + src_off[ti] + kk*ctL and its two outputs go to dst_off[ti] + {kk, kk + 2^j}*ctL.
struct LevelArgs {
  const u64* src_off;  // device, [n_trees] limb offsets
  const u64* dst_off;  // device, [n_trees]
  int n_trees;
  int j;         // tree level; 2^j nodes per tree
  u32 ginv;      // inverse of the Galois element (N>>j)+1 modulo 2N
  u32 g;         // the Galois element itself
  u64 q_stride;  // limbs between consecutive queries' workspaces
  int n_queries;
  // per-query Galois keys (queries of different clients in one launch): device array of n_queries key pointers of
  // this level, entry qi for query qi of the launch; nullptr: every node uses the launch's `key` argument.  Complete
  // before the call's first kernel starts (the cluster kernels read it before griddepcontrol.wait).
  const u64* const* key_tab;
  u64* xch;      // cluster kernel: [node][2][N] scratch through which the special-prime accumulators reach the
                 // other CTAs of the cluster (L2 moves them faster than distributed shared memory does)
  u64* dbg;      // optional per-CTA phase timestamps (clock64), 8 slots per CTA; nullptr in production
  int dbg_clock; // 1: slots 0 and 7 are clock64 too (single-level probe); 0: globaltimer (level-to-level gaps)
};

// generic batched transforms on [n_polys][N] arrays; modulus of poly p is m[(p % cycle) + off].
// inverse sums n_parts partial inputs (stride part_stride limbs) mod q before transforming.
cudaError_t launch_ntt_fwd(const DevParams& P, const u64* in, u64* out, int n_polys, int cycle, int off,
                           int n_batch, u64 in_bstride, u64 out_bstride, cudaStream_t st);
cudaError_t launch_ntt_inv(const DevParams& P, const u64* in, u64* out, int n_polys, int cycle, int off, int n_parts,
                           u64 part_stride, int n_batch, u64 in_bstride, u64 out_bstride, cudaStream_t st);

// plaintext coefficients (< t, [n_pt][N]) -> centred lift -> NTT per data modulus -> [n_pt][k][N]
cudaError_t launch_db_preprocess(const DevParams& P, const u64* coeffs, u64* out, u64 n_pt, cudaStream_t st);

// key switching, step 1: sigma_g(c1) digit J re-reduced mod m_I and forward-transformed -> dig[z][I][J][N]
cudaError_t launch_ks_digits(const DevParams& P, const u64* work, const LevelArgs& L, u64* dig, cudaStream_t st);
// step 2: acc[z][c][I] = INTT_I( sum_J dig[z][I][J] (.) key[J][c][I] ); with key_tab, node z uses
// key_tab[z / nodes_per_query] instead of key
cudaError_t launch_ks_mac_intt(const DevParams& P, const u64* dig, const u64* key, u64* acc, int n_nodes,
                               cudaStream_t st, const u64* const* key_tab = nullptr, u32 nodes_per_query = 1);
// step 3: mod-down by P with rounding + (mode 0) SealPIR expansion combine / (mode 1) plain substitution result
cudaError_t launch_ks_combine(const DevParams& P, u64* work, const LevelArgs& L, const u64* acc, int mode,
                              cudaStream_t st);

// all three steps in one launch: a thread-block cluster of 2(k+1) CTAs per node, digits and accumulators stay in
// (distributed) shared memory (kernels_cluster.cu)
bool ks_cluster_supported(const DevParams& P);
cudaError_t launch_ks_level_cluster(const DevParams& P, u64* work, const LevelArgs& L, const u64* key, int mode,
                                    cudaStream_t st);

// ct * x^{-kpow}  (server.cpp:78-103)
cudaError_t launch_mul_inv_pow_x(const DevParams& P, const u64* in, u64* out, u32 kpow, int n_cts, cudaStream_t st);

// last-dimension inner product against the HBM-resident database (SURVEY §3.1 HOT LOOP 2)
// part[qi][split][row][2][k][N] = sum over the split's share of i1 of sv[qi][i1] (.) db[row*dimL + i1]   (mod q)
cudaError_t launch_scan(const DevParams& P, const u64* db, u64 num_pt, u32 dimL, u32 n_rows, const u64* sv,
                        u64 sv_qstride, int n_queries, int n_split, u64* part, cudaStream_t st);
void scan_config(const DevParams& P, u32 dimL, u32 n_rows, int n_queries, int sm_count, int* n_split);

// re-encode (ct_reencoder.cpp:40-71) + centred lift + forward NTT: cts [n_cts][2][k][N] -> pts [n_cts][2ER][k][N]
cudaError_t launch_reencode_ntt(const DevParams& P, const u64* cts, u64* pts, int n_cts, cudaStream_t st);

// upper-dimension MAC (SURVEY §3.1 HOT LOOP 3):
// part[qi][split][g][x][2][k][N] = sum_{i in split, i < cnt(g)} sv[qi][i][c] (.) pts[qi][(g*dim+i)][x]
int dim_mac_config(const DevParams& P, u64 base_ctas, u32 len, int sm_count);  // n_split for launch_dim_mac
cudaError_t launch_dim_mac(const DevParams& P, const u64* pts, u64 pts_qstride, const u64* sv, u64 sv_qstride,
                           int n_queries, u32 dim, u32 n_entries_in, u32 n_groups, u32 w_out, int n_split, u64* part,
                           cudaStream_t st);

// out[i] = sum_g in[g*stride + i] mod q_j(i)   for [n_cts][2][k][N] arrays (cross-GPU partial combine)
// (n_batch independent reductions, in_bstride / out_bstride limbs apart)
cudaError_t launch_modadd_reduce(const DevParams& P, const u64* in, u64 stride, int n_parts, u64* out, u64 n_cts,
                                 cudaStream_t st, int n_batch = 1, u64 in_bstride = 0, u64 out_bstride = 0);
// out[i] = sum over peers of *(peers[g] + i) mod q: same, reading each partial through its own (peer) pointer
cudaError_t launch_modadd_reduce_ptrs(const DevParams& P, const u64* const* peers_dev, int n_parts, u64 offset_limbs,
                                      u64* out, u64 n_cts, cudaStream_t st);

// copy root ciphertexts of every tree into place: work[qi*q_stride + root_off[t]] = query[qi][t]
cudaError_t launch_place_roots(const DevParams& P, const u64* query, u64 query_qstride, u64* work, const u64* root_off,
                               int n_trees, int n_queries, u64 q_stride, cudaStream_t st);

// ---- cross-GPU exchange over NVLink peer memory (kernels_dist.cu) ----
// Every rank owns one exchange block (flags, selection-vector slots, partial-reply slots) that all peers map.
struct PushArgs {
  u64* const* peers;   // device array [n_ranks]: base pointers of the ranks' exchange blocks (own included)
  u32 n_ranks;
  u32 d0;              // dims[0]
  u32 rows_per_rank;   // ceil(d0 / n_ranks): rank r owns rows [r * rows_per_rank, ...) of the first dimension
  u64 slot_off;        // limb offset of the destination slot inside every rank's block
  u64 g_first;         // position of this launch's first query in the slot's query order
  u64 dst_qstride;     // limbs per query in the slot
};
// forward NTT of the first n_entries selection ciphertexts of n_queries queries (in: coefficient form, in_qstride limbs
// apart) with the outputs stored into the peers' slots in the compact layout [own rows of dim 0 | dims 1..]
cudaError_t launch_ntt_fwd_push(const DevParams& P, const u64* in, u64 in_qstride, u32 n_entries, u32 n_queries,
                                const PushArgs& A, cudaStream_t st);
// copy-only variant for selection vectors that are already in NTT form (n_entries leading entries of n_queries queries)
cudaError_t launch_push_head(const DevParams& P, const u64* in, u64 in_qstride, u32 n_entries, u32 n_queries,
                             const PushArgs& A, cudaStream_t st);
// The last-dimension entries only feed the scan.  When that runs on the tensor cores they travel already repacked into
// its operand layout (svT, kernels_tc.cu): the producing rank packs its own queries once into a staging buffer
// [coefficient][rows][Kp] (src_stride bytes per coefficient) and this kernel copies every coefficient's segment (seg_bytes) into every
// peer's svT region at dst_off + coefficient * dst_stride (bytes from the peer's block base).  Narrow grid, 16-byte
// loads and stores: the copy drains at NVLink speed.
cudaError_t launch_push_rows(u64* const* peers_dev, u32 n_ranks, const u8* stage, u64 src_stride, u32 seg_bytes, u32 n_segs,
                             u64 dst_off, u64 dst_stride, cudaStream_t st);
// flag[off] = value in every rank's block (release, system scope), ordered after the stream's earlier kernels
cudaError_t launch_signal(u64* const* peers_dev, u32 n_ranks, u64 flag_off_limbs, u64 value, cudaStream_t st);
// spin until flags[0..n_ranks) >= value (acquire, system scope); after timeout_ns sets *err and returns
cudaError_t launch_wait(const u64* flags, u32 n_ranks, u64 value, u64 timeout_ns, u64* err, cudaStream_t st);

// ---- batched scan on the tensor cores (kernels_tc.cu) ----
struct TcGeom {
  u32 nb;       // byte limbs per residue (5 or 6)
  u32 rpt;      // database rows per 128-lane MMA tile = 128 / nb
  u32 ntiles;   // MMA tiles per coefficient slot
  u32 Kp;       // dimL rounded up to a multiple of 16 (TMA row pitch)
  u32 kch;      // 128-byte K chunks
  u64 db_bytes; // size of the byte-planar database copy
};
// launch plan (tc_plan.h) of a scan of n_queries queries over a last dimension of dimL entries, with the query tile
// requested by PIRB_TC_QT; false when the device or the moduli rule the tensor cores out or no plan fits
bool tc_launch_plan(const DevParams& P, u32 dimL, u32 n_queries, TcPlan* plan);
void tc_geometry(const DevParams& P, u32 dimL, u32 n_rows, TcGeom* g);
u64 tc_sv_bytes(const DevParams& P, const TcGeom& g, const TcPlan& plan);
// u64 database [pt][k][N] -> byte-planar K-major copy dbT (db_bytes)
cudaError_t launch_tc_pack_db(const DevParams& P, const u64* db, u64 num_pt, u32 dimL, u32 n_rows, const TcGeom& g,
                              u8* dbT, cudaStream_t st);
// part[q][row][2][k][N] = sum_i1 sv[q][i1] (.) db[row*dimL + i1] mod q for a batch of queries (svT: scratch of
// tc_sv_bytes; err_flag: device-visible int raised if the kernel's internal pipeline times out)
// pack + scan for selection vectors held as u64 limbs [q][i1][2][k][N] (sv_qstride limbs between queries); svT: scratch
// of tc_sv_bytes; plan: tc_launch_plan for n_queries
cudaError_t launch_tc_scan(const DevParams& P, const TcGeom& g, const TcPlan& plan, const u8* dbT, u32 dimL, u32 n_rows,
                           const u64* sv, u64 sv_qstride, u32 n_queries, u8* svT, int* err_flag, int sm_count, u64* part,
                           cudaStream_t st);
// the two halves: repack n_queries selection vectors into rows [row0, row0 + n_queries*2*nb) of an svT array with
// rows_total rows per coefficient; scan against an svT array whose rows [row0, ...) hold the n_queries queries
cudaError_t launch_tc_pack_sv(const DevParams& P, const TcGeom& g, const u64* sv, u64 sv_qstride, u32 dimL, u32 n_queries,
                              u8* svT, u32 rows_total, u32 row0, cudaStream_t st);
cudaError_t launch_tc_scan_packed(const DevParams& P, const TcGeom& g, const TcPlan& plan, const u8* dbT, u32 n_rows,
                                  const u8* svT, u32 rows_total, u32 row0, u32 n_queries, int* err_flag, int sm_count,
                                  u64* part, cudaStream_t st);

// ---- ciphertext-multiplication mode (kernels_ctmul.cu; database.cpp:202-211) ----
// Evaluator::multiply [SEAL 3.5.6 bfv_multiply, BEHZ] split at its NTTs; n_batch independent problems, *_bstride apart.
// (1)-(2) base q -> Bsk: in [n_polys][k][N] -> out [n_polys][nB+1][N], coefficient form
cudaError_t launch_behz_extend(const BehzC& B, const u64* in, u64 in_bstride, u32 n_polys, u64* out, u64 out_bstride,
                               int n_batch, cudaStream_t st);
// (4) D[e][s1+1] = A[e][s1] (x) S[e % dim][2] in base q (base = 0) or Bsk (base = 1), NTT form
cudaError_t launch_behz_tensor(const BehzC& B, int base, const u64* A, u64 a_bstride, const u64* S, u64 s_bstride, u64* D,
                               u64 d_bstride, u32 n_entries, u32 dim, int s1, int n_batch, cudaStream_t st);
// (6)-(8) scale by t/Q and round: Dq [n_polys][k][N], Db [n_polys][nB+1][N] -> out [n_polys][k][N], coefficient form
cudaError_t launch_behz_floor(const BehzC& B, const u64* Dq, u64 dq_bstride, const u64* Db, u64 db_bstride, u64* out,
                              u64 out_bstride, u32 n_polys, int n_batch, cudaStream_t st);
// Evaluator::relinearize_inplace of n_entries size-3 products prod [e][3][k][N]:
// digits [e][J][I][N] (then forward NTT, cycle k+1) -> mac with the key -> acc [e][2][k+1][N] (then inverse NTT)
// -> finish: X [e][2][k][N]
cudaError_t launch_relin_digits(const BehzC& B, const u64* prod, u64 p_bstride, u64* dig, u64 dig_bstride, u32 n_entries,
                                int n_batch, cudaStream_t st);
cudaError_t launch_relin_mac(const BehzC& B, const u64* dig, u64 dig_bstride, const u64* key, u64* acc, u64 acc_bstride,
                             u32 n_entries, int n_batch, cudaStream_t st);
cudaError_t launch_relin_finish(const BehzC& B, const u64* prod, u64 p_bstride, const u64* acc, u64 acc_bstride, u64* X,
                                u64 x_bstride, u32 n_entries, int n_batch, cudaStream_t st);
// out [g][polys][k][N] = sum over the entries of group g (dim per group, the last one may be short) of X [e][polys][k][N]
cudaError_t launch_ct_reduce(const BehzC& B, const u64* X, u64 x_bstride, u64* out, u64 out_bstride, u32 n_entries, u32 dim,
                             u32 polys, int n_batch, cudaStream_t st);

// StringEncoder packing on the device: raw item bytes -> plaintext coefficients [n_pt][N]
cudaError_t launch_pack_items(const u8* bytes, u64* coeffs, u32 N, u32 bits, u64 bytes_per_pt, u64 total_bytes,
                              u64 n_pt, cudaStream_t st);

// warm L2 with constants that every kernel of a query re-reads (tables, keys)
cudaError_t launch_prefetch_l2(const void* p, u64 bytes, cudaStream_t st);

// synthetic data: out[p][N] uniform in [0, q_{(p % cycle) + off}) from a counter-based generator keyed by the global
// polynomial index poly0 + p (poly0 must be a multiple of cycle)
cudaError_t launch_fill_random(const DevParams& P, u64* out, u64 n_polys, int cycle, int off, u64 seed, u64 poly0,
                               cudaStream_t st);

}  // namespace pirb
