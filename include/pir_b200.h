/* pir_b200.h — C ABI of the B200-native PIR server answer path.
 *
 * Drop-in boundary for OpenMined/PIR's server side.  The reference has no FFI layer; its boundary is the
 * public C++ API of pir::PIRServer / pir::PIRDatabase (pir/cpp/server.h:43-131, pir/cpp/database.h:47-127).
 * Each entry point below cites the reference interface it replaces.  All ciphertext / plaintext / key
 * arguments are raw RNS limbs, uint64, values in [0, q_j), laid out exactly as SEAL lays them out in
 * Ciphertext::data(i) (the reference relies on that layout directly: server.cpp:94-100,
 * ct_reencoder.cpp:58-63):
 *
 *   ciphertext  [2][k][N]            poly-major, then RNS modulus, then coefficient        (ct_limbs = 2kN)
 *   plaintext   [N] coefficients < t (coefficient form)   or   [k][N] (NTT form)           (pt_limbs = kN)
 *   Galois key  [k][2][k+1][N]       digit J, component c, key-level modulus I, NTT form    (key_limbs)
 *               == seal::KSwitchKeys::data()[index][J].data().data(c)[I*N + n]
 *
 * NTT form uses SEAL's ordering (minimal primitive 2N-th root, bit-reversed output) so keys and
 * preprocessed databases produced by SEAL can be loaded unchanged.
 *
 * Status codes follow absl::StatusCode as the reference uses it: 0 OK, 3 InvalidArgument, 13 Internal.
 * pirb_last_error() returns the message of the last failure on the calling thread.
 * A context may be used from one host thread at a time; batching is explicit (n_queries).
 * There is NO CPU fallback: every entry point that computes fails with 13 if CUDA is unavailable.
 */
#ifndef PIR_B200_H_
#define PIR_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PIRB_OK 0
#define PIRB_INVALID_ARGUMENT 3
#define PIRB_INTERNAL 13

#define PIRB_MAX_MODULI 9
#define PIRB_MAX_DIMS 8

typedef struct pirb_ctx pirb_ctx;   /* owns device tables, the HBM-resident database shard, workspaces, a stream */
typedef struct pirb_keys pirb_keys; /* one client's Galois keys, resident in HBM */

/* What PIRContext::Create / PIRParameters carry for this path (pir/cpp/context.cpp:37-50,
 * pir/proto/payload.proto:45-69), with the SEAL EncryptionParameters unpacked. */
typedef struct {
  uint32_t poly_modulus_degree;               /* N, power of two, 2048..16384 */
  uint32_t n_moduli;                          /* k+1: data-level primes q_0..q_{k-1}, then the special prime P */
  uint64_t coeff_modulus[PIRB_MAX_MODULI];
  uint64_t plain_modulus;                     /* t */
  uint32_t n_dims;                            /* d */
  uint32_t dims[PIRB_MAX_DIMS];               /* PIRParameters.dimensions */
  uint64_t num_pt;                            /* PIRParameters.num_pt (whole database, all shards) */
  int32_t device;                             /* CUDA device ordinal */
  uint32_t shard_index;                       /* row shard of dims[0] owned by this context ... */
  uint32_t shard_count;                       /* ... out of shard_count (1 = whole database) */
  uint32_t use_ciphertext_multiplication;     /* PIRParameters.use_ciphertext_multiplication (payload.proto:69): upper
                                               * dimensions by Evaluator::multiply instead of the re-encoder
                                               * (database.cpp:202-211); one GPU, entry points pirb_*_ct below */
} pirb_params;

const char* pirb_last_error(void);

/* PIRServer::Create + PIRContext::Create (server.cpp:35-42, context.cpp:37-50). */
int pirb_ctx_create(const pirb_params* params, pirb_ctx** out);
void pirb_ctx_destroy(pirb_ctx* ctx);

/* shape queries */
uint64_t pirb_ct_limbs(const pirb_ctx* ctx);
uint64_t pirb_pt_limbs(const pirb_ctx* ctx);
uint64_t pirb_key_limbs(const pirb_ctx* ctx);
uint32_t pirb_expansion_ratio(const pirb_ctx* ctx);      /* CiphertextReencoder::ExpansionRatio (ct_reencoder.cpp:29-38) */
uint64_t pirb_reply_cts(const pirb_ctx* ctx);            /* (2*ER)^(d-1)  (database.cpp:215, client.cpp:224-226) */
uint64_t pirb_dim_sum(const pirb_ctx* ctx);              /* PIRContext::DimensionsSum (context.h:59-62) */
uint64_t pirb_query_cts(const pirb_ctx* ctx);            /* dim_sum / N + 1 (client.cpp:109, server.cpp:154-158) */
uint64_t pirb_shard_pt_begin(const pirb_ctx* ctx);       /* first plaintext index held by this shard */
uint64_t pirb_shard_pt_count(const pirb_ctx* ctx);
uint64_t pirb_db_size(const pirb_ctx* ctx);              /* PIRDatabase::size(): plaintexts loaded so far (database.h:94) */

/* PIRDatabase::populate (database.cpp:84-110) after StringEncoder/IntegerEncoder packing:
 * coeffs[count][N] < t, plaintext indices are GLOBAL; the shard keeps the ones it owns.
 * The centred lift + NTT (transform_to_ntt_inplace(pt, first_parms_id), database.cpp:103-106) run on the GPU. */
int pirb_db_load_coeff(pirb_ctx* ctx, const uint64_t* coeffs, uint64_t first_pt, uint64_t count);
/* PIRDatabase::populate(vector<string>) entirely on the device: `items` holds n_items raw items of bytes_per_item
 * bytes each, starting at GLOBAL item index first_item (which must start a plaintext).  StringEncoder's MSB-first bit
 * packing (string_encoder.cpp:58-80, 108-122; bits_per_coeff = 0 means trunc(log2 t)), the centred lift and the NTT all
 * run on the GPU; only the raw bytes cross PCIe. */
int pirb_db_load_items(pirb_ctx* ctx, const uint8_t* items, uint64_t first_item, uint64_t n_items,
                       uint32_t bytes_per_item, uint32_t items_per_plaintext, uint32_t bits_per_coeff);
/* Same, for a database already in NTT form (SEAL ordering): limbs[count][k][N]. */
int pirb_db_load_ntt(pirb_ctx* ctx, const uint64_t* limbs, uint64_t first_pt, uint64_t count);
/* Read back NTT-form plaintexts (persistence / tests): out[count][k][N]. */
int pirb_db_read_ntt(const pirb_ctx* ctx, uint64_t* out, uint64_t first_pt, uint64_t count);
/* Synthetic database for benchmarks: uniform limbs in [0,q_j), generated on the device (scan cost is data-independent). */
int pirb_db_fill_random(pirb_ctx* ctx, uint64_t seed);

/* seal::GaloisKeys as deserialized by ProcessRequest (server.cpp:46-48): n keys, elts[i] = Galois element. */
int pirb_keys_load(pirb_ctx* ctx, const uint32_t* elts, uint32_t n_elts, const uint64_t* limbs, pirb_keys** out);
void pirb_keys_destroy(pirb_keys* keys);

/* PIRServer::substitute_power_x_inplace (server.cpp:67-76): ct(x) -> ct(x^power), in place. 13 if the key is missing. */
int pirb_substitute(pirb_ctx* ctx, const pirb_keys* keys, uint64_t* ct, uint32_t power);
/* PIRServer::multiply_inverse_power_of_x (server.cpp:78-103). */
int pirb_mul_inv_pow_x(pirb_ctx* ctx, const uint64_t* ct_in, uint32_t k, uint64_t* ct_out);
/* PIRServer::oblivious_expansion: single != 0 -> the one-ciphertext overload (server.cpp:105-146), else the
 * vector overload (server.cpp:148-171).  out[total_items][2][k][N].  3 on the reference's argument errors. */
int pirb_expand(pirb_ctx* ctx, const pirb_keys* keys, const uint64_t* cts, uint64_t n_ct, uint64_t total_items,
                int single, uint64_t* out);
/* PIRDatabase::multiply (database.cpp:290-316), re-encoder path.  sv[n_sv][2][k][N] in coefficient form is
 * transformed to NTT form IN PLACE like the reference does (database.cpp:190,222).  out[(2*ER)^(d-1)][2][k][N].
 * 3 if n_sv != dim_sum. */
int pirb_db_multiply(pirb_ctx* ctx, uint64_t* sv, uint64_t n_sv, uint64_t* out, uint64_t out_cap_cts,
                     uint64_t* out_count);
/* PIRServer::processQuery for every query of a request (server.cpp:60-63, 173-195): expansion + multiply.
 * queries[n_queries][n_ct][2][k][N] -> replies[n_queries][reply_cts][2][k][N].  Host buffers; page-locked ones
 * (cudaHostAlloc / cudaHostRegister) are read and written in place by the kernels, pageable ones are staged. */
int pirb_answer(pirb_ctx* ctx, const pirb_keys* keys, const uint64_t* queries, uint32_t n_queries, uint64_t n_ct,
                uint64_t* replies);
/* PIRServer::processQuery for queries of several clients in one pass: keys[i] is the Galois-key handle of query i
 * (handles may repeat, in any order).  Same buffers, layouts, status codes and zero-copy rules as pirb_answer /
 * pirb_answer_dev.  Unsharded, re-encoder contexts only (3 otherwise).  Every handle is checked before anything runs:
 * 3 for a null handle or one loaded on a context of another shape, 13 for a handle that lacks the Galois element of
 * an expansion level; the message names the query, and no reply is written.  pirb_answer_multi_dev returns before the
 * device has read the handles' keys: the caller must not destroy a handle while such a call that uses it is in flight. */
int pirb_answer_multi(pirb_ctx* ctx, const pirb_keys* const* keys, const uint64_t* queries, uint32_t n_queries,
                      uint64_t n_ct, uint64_t* replies);

/* ---- Ciphertext-multiplication mode (PIRParameters.use_ciphertext_multiplication; contexts created with the flag).
 * The upper dimensions multiply the lower result with the selection ciphertext by Evaluator::multiply and, when the
 * request carries relinearization keys, Evaluator::relinearize_inplace (database.cpp:202-211, server.cpp:185-190)
 * [SEAL 3.5.6: BEHZ RNS multiplication, switch_key_inplace].  The reply of a query is ONE ciphertext
 * (client.cpp:196-217) of pirb_reply_polys polynomials: 2 with relinearization keys (or d = 1), else d + 1.
 * The entry points above that multiply (pirb_db_multiply, pirb_answer*, pirb_dist_*) fail with 3 on such a context. */
/* seal::RelinKeys as KeyGenerator::relin_keys() makes them (client.cpp:49): one key-switching key (for s^2),
 * limbs [k][2][k+1][N] in NTT form — the layout of one Galois key.  Freed with pirb_keys_destroy. */
int pirb_relin_keys_load(pirb_ctx* ctx, const uint64_t* limbs, pirb_keys** out);
uint32_t pirb_reply_polys(const pirb_ctx* ctx, int with_relin_keys);
/* PIRDatabase::multiply(selection_vector, relin_keys) (database.cpp:290-316).  sv[n_sv][2][k][N] in coefficient form
 * is NOT modified (database.cpp:188 only transforms it on the re-encoder path).  relin may be NULL.
 * out[polys][k][N]; *out_polys = polys (0 for an empty database).  3 if n_sv != dim_sum. */
int pirb_db_multiply_ct(pirb_ctx* ctx, const uint64_t* sv, uint64_t n_sv, const pirb_keys* relin, uint64_t* out,
                        uint64_t out_cap_limbs, uint32_t* out_polys);
/* PIRServer::processQuery with optional<RelinKeys> for every query of a request (server.cpp:60-63, 173-195).
 * queries[n_queries][n_ct][2][k][N] -> replies[n_queries][polys][k][N].  Host buffers. */
int pirb_answer_ct(pirb_ctx* ctx, const pirb_keys* galois_keys, const pirb_keys* relin, const uint64_t* queries,
                   uint32_t n_queries, uint64_t n_ct, uint64_t* replies);

/* Device-resident variants (pointers are CUDA device pointers on ctx's device; stream = cudaStream_t or NULL
 * for the context's own stream).  pirb_answer_dev writes final replies (shard_count == 1).  With shards, each rank
 * calls pirb_answer_partial_dev -> partial[n_queries][reply_cts][2][k][N] in NTT form (sum over its rows), the
 * partials are exchanged by NCCL all-gather and pirb_reduce_finish_dev adds them mod q and applies the final inverse
 * NTT (database.cpp:250-254).  A plain integer sum is never used. */
int pirb_answer_dev(pirb_ctx* ctx, const pirb_keys* keys, const uint64_t* d_queries, uint32_t n_queries,
                    uint64_t n_ct, uint64_t* d_replies, void* stream);
int pirb_answer_partial_dev(pirb_ctx* ctx, const pirb_keys* keys, const uint64_t* d_queries, uint32_t n_queries,
                            uint64_t n_ct, uint64_t* d_partial, void* stream);
/* pirb_answer_dev with one Galois-key handle per query (see pirb_answer_multi) */
int pirb_answer_multi_dev(pirb_ctx* ctx, const pirb_keys* const* keys, const uint64_t* d_queries, uint32_t n_queries,
                          uint64_t n_ct, uint64_t* d_replies, void* stream);
/* The two halves of pirb_answer_partial_dev, for batches whose expansion is split by query across ranks:
 * pirb_expand_ntt_dev: oblivious expansion (server.cpp:148-171) + the selection-vector NTT (database.cpp:190,222)
 *   -> d_sv_ntt[n_queries][dim_sum][2][k][N];
 * pirb_multiply_partial_dev: scan + re-encode + upper dimensions of this shard's rows for NTT-form selection
 *   vectors (own and all-gathered ones) -> d_partial[n_queries][reply_cts][2][k][N], NTT form. */
int pirb_expand_ntt_dev(pirb_ctx* ctx, const pirb_keys* keys, const uint64_t* d_queries, uint32_t n_queries,
                        uint64_t n_ct, uint64_t* d_sv_ntt, void* stream);
int pirb_multiply_partial_dev(pirb_ctx* ctx, const uint64_t* d_sv_ntt, uint32_t n_queries, uint64_t* d_partial,
                              void* stream);
int pirb_reduce_finish_dev(pirb_ctx* ctx, const uint64_t* d_partials, uint32_t n_parts, uint64_t part_stride_limbs,
                           uint32_t n_queries, uint64_t* d_replies, void* stream);
/* Row-sharded serving with the exchange done by the kernels themselves over NVLink peer memory (SURVEY §8e; replaces
 * the NCCL gathers of the flow above for databases of d >= 2 dimensions).  Every rank (= context with shard_index r of
 * shard_count) owns ONE exchange block — flags, two selection-vector slots, two partial-reply slots — that all peers
 * map.  pirb_dist_create allocates it (max_local_queries = queries a rank brings to a step; sub_batch = local queries
 * per pipelined sub-batch, 0 = default) and returns its CUDA IPC handle (ranks in separate processes: exchange the
 * handles, then pirb_dist_open_ipc) and its base pointer (contexts of one process on peer-accessible devices:
 * pirb_dist_attach with everybody's base pointers).  pirb_dist_answer* then runs one step: this rank's n_local
 * queries (ALL ranks must call it with the same n_local, in lockstep) -> this rank's replies.  The rank expands its own
 * queries; the selection-vector NTT kernel stores its output directly into every peer's slot (first-dimension entries
 * only at the row's owner) and raises per-sub-batch flags; every rank multiplies all ranks' queries against its rows
 * as soon as a sub-batch has arrived from everyone; the partial replies are added mod q by loads from the peers'
 * partial slots inside the reduce kernel and go through the final inverse NTT (database.cpp:250-254).  A flag that
 * does not arrive within the timeout (PIRB_DIST_TIMEOUT_MS, default 20 s) makes pirb_dist_status return 13. */
int pirb_dist_create(pirb_ctx* ctx, uint32_t max_local_queries, uint32_t sub_batch, uint8_t* ipc_handle_out /*[64] or NULL*/,
                     void** base_out /* or NULL */);
int pirb_dist_open_ipc(pirb_ctx* ctx, const uint8_t* ipc_handles /*[n_ranks][64]*/, uint32_t n_ranks, uint32_t self_rank);
int pirb_dist_attach(pirb_ctx* ctx, void* const* peer_bases /*[n_ranks]*/, uint32_t n_ranks, uint32_t self_rank);
/* Optional, needed when several ranks are driven by ONE host thread (contexts of one process): sizes every workspace
 * for steps of n_local queries and runs one warm-up step in which the rank exchanges only with itself, so that no
 * allocation, module load or attribute change (all of which may synchronise the device) happens between one rank's
 * wait for a flag and the launches of the rank that raises it.  Call it on every rank before the first step. */
int pirb_dist_prepare(pirb_ctx* ctx, const pirb_keys* keys, uint32_t n_local);
/* device-accessible buffers, asynchronous on `stream` (NULL: the context's stream) */
int pirb_dist_answer_dev(pirb_ctx* ctx, const pirb_keys* keys, const uint64_t* d_queries, uint32_t n_local, uint64_t n_ct,
                         uint64_t* d_replies, void* stream);
/* host buffers (page-locked ones are used in place), synchronous; returns pirb_dist_status */
int pirb_dist_answer(pirb_ctx* ctx, const pirb_keys* keys, const uint64_t* queries, uint32_t n_local, uint64_t n_ct,
                     uint64_t* replies);
int pirb_dist_status(pirb_ctx* ctx);
/* device times of the last profiled step: 0 expansion, 1 exchange tail after the expansion, 2 start -> first sub-batch
 * of every rank has arrived, 3 multiplies, 4 partial-reply reduce + inverse NTT, 5 whole step */
int pirb_dist_stage_ms(pirb_ctx* ctx, float* out_ms /*[10]: the six above, then the transfer stream's phases for the last
                                                      sub-batch: selection-vector NTT, first-dimension push, repack, row push */);

/* Scan only (the HBM-bound kernel): d_sv_ntt[n_queries][dims[d-1]][2][k][N] NTT form -> rows in NTT form.
 * Used by the bench to time the scan in isolation.  d_rows may be NULL (internal scratch). */
int pirb_scan_dev(pirb_ctx* ctx, const uint64_t* d_sv_ntt, uint32_t n_queries, uint64_t* d_rows, void* stream);
int pirb_sync(pirb_ctx* ctx);
/* development aid: clock64 phase stamps of one expansion level (env PIRB_DEBUG_STAMPS=<level> at context creation) */
int pirb_debug_stamps(pirb_ctx* ctx, uint64_t* out, uint64_t n);

/* Per-stage device times of the last pirb_answer* call, measured with CUDA events on the launching stream
 * when profiling is enabled.  stage: 0 expand, 1 sv NTT, 2 scan, 3 row INTT, 4 upper dims, 5 total. */
#define PIRB_N_STAGES 6
int pirb_set_profiling(pirb_ctx* ctx, int enabled);
int pirb_get_stage_ms(pirb_ctx* ctx, float* out_ms /*[PIRB_N_STAGES]*/);
/* device time of the scan kernel of the last profiled pirb_scan_dev / pirb_answer* call */
int pirb_last_scan_ms(pirb_ctx* ctx, float* out_ms);
/* kernels launched by the last pirb_answer* call, and algorithmic scan bytes of one scan launch (SURVEY §8d). */
uint64_t pirb_last_launch_count(const pirb_ctx* ctx);
uint64_t pirb_scan_bytes(const pirb_ctx* ctx, uint32_t n_queries);

/* Page-locked host memory (portable across devices, mapped): buffers from here are read and written IN PLACE by the
 * kernels of pirb_answer / pirb_dist_answer* — no staging copies — and keep the captured CUDA graphs of pirb_answer
 * valid across calls (they are keyed on the buffer addresses).  For hosts that do not link the CUDA runtime. */
int pirb_host_alloc(uint64_t bytes, void** out);
void pirb_host_free(void* p);

/* Host-side shape math of the reference, exported so bindings need not re-implement it:
 * PIRDatabase::calculate_dimensions (database.cpp:334-342), next_power_two / ceil_log2 / log2 (utils.h:29-37,
 * utils.cpp:16-44), PlainModulus::Batching and CoeffModulus::BFVDefault as used by GenerateEncryptionParams
 * (parameters.cpp:33-54). */
void pirb_calculate_dimensions(uint32_t db_size, uint32_t n_dims, uint32_t* out);
uint64_t pirb_next_power_two(uint64_t v);
uint32_t pirb_ceil_log2(uint32_t v);
uint32_t pirb_log2(uint32_t v);
uint64_t pirb_plain_modulus_batching(uint32_t poly_modulus_degree, uint32_t bit_size);
int pirb_bfv_default_coeff_modulus(uint32_t poly_modulus_degree, uint64_t* out, uint32_t cap);

#ifdef __cplusplus
}
#endif
#endif /* PIR_B200_H_ */
