/* include/seal_b200.h -- C-ABI of libseal_b200.so: the B200 (sm_100a) drop-in for the RNS-polynomial hot path of
 * microsoft/SEAL 4.4.3 (negacyclic NTT/INTT, dyadic products, hybrid key switching, rescale / BEHZ base conversion)
 * that backs Evaluator::multiply / relinearize_inplace / rotate_rows / rotate_vector / rescale_to_next.
 *
 * Style follows the reference's own C layer (native/src/seal/c/defines.h:34-96): extern "C", opaque handles, plain
 * pointers and sizes, an integer status instead of exceptions, a last-error string.  Unlike the reference's C layer
 * the data arguments are raw uint64 slabs laid out exactly like seal::Ciphertext::data() (ciphertext.h:24-37):
 *
 *      [batch][poly (size)][rns prime (L)][coefficient (n)]       8*n*L*size bytes per ciphertext
 *
 * so a binding marshals `ct.data()` with one memcpy (see INTEGRATION.md).  `L` = number of RNS primes the
 * ciphertexts carry = parms.coeff_modulus().size() at that level of the modulus-switching chain; the key level has
 * k primes, ciphertexts have L <= k-1 (context.cpp:513-535).  Device entry points (d_ prefix on arguments) are
 * stream-ordered and never synchronise; the *_host entry points take host buffers, copy H2D / D2H themselves and
 * return after the result is in the host buffer.
 *
 * There is NO CPU fallback: every entry point fails with SB200_E_CUDA when no sm_100 device is usable.
 */
#ifndef SEAL_B200_H
#define SEAL_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

/* status codes; the mapping mirrors the reference's exception -> HRESULT ladder (c/defines.h:72-96) */
#define SB200_OK 0
#define SB200_E_INVALID_ARG (-1)  /* std::invalid_argument  -> E_INVALIDARG            */
#define SB200_E_LOGIC (-2)        /* std::logic_error       -> COR_E_INVALIDOPERATION  */
#define SB200_E_OUT_OF_RANGE (-3) /* std::out_of_range      -> ERROR_INVALID_INDEX     */
#define SB200_E_CUDA (-4)         /* std::runtime_error     -> COR_E_IO                */
#define SB200_E_NOMEM (-5)        /* std::bad_alloc         -> E_OUTOFMEMORY           */
#define SB200_E_POINTER (-6)      /* null handle / pointer  -> E_POINTER               */

#define SB200_SCHEME_BFV 1  /* seal::scheme_type::bfv  (encryptionparams.h) */
#define SB200_SCHEME_CKKS 2 /* seal::scheme_type::ckks */
#define SB200_SCHEME_BGV 3  /* seal::scheme_type::bgv: NTT-form ciphertexts like CKKS, plain-modulus-aware mod-down (SURVEY 8f rank 2) */

typedef struct sb200_context sb200_context;   /* mirrors SEALContext + Evaluator state (context.h:277-439) */
typedef struct sb200_public_key sb200_public_key;   /* Encryptor state: the public key on the device (publickey.h) */
typedef struct sb200_secret_key sb200_secret_key;   /* Decryptor state: the secret key and its powers on the device (decryptor.h) */
typedef struct sb200_kswitch_key sb200_kswitch_key; /* one KSwitchKeys::data()[index] entry on the device (kswitchkeys.h) */

/* last error message of the calling thread (never NULL) */
const char *sb200_last_error(void);

/* ---- context ------------------------------------------------------------------------------------------------
 * Replaces SEALContext(parms, expand_mod_chain=true, sec_level_type::none) + Evaluator(context) for this path
 * (context.cpp:495-563, evaluator.cpp:121-128).  coeff_modulus = the k key-level primes (last = special prime),
 * each < 2^61, prime, = 1 mod 2n.  plain_modulus is used by BFV and BGV (BGV: coprime to every prime, rns.cpp:778-787).  All NTT / RNS / Galois tables are computed
 * here from these numbers alone and uploaded to CUDA device `device`. */
int sb200_context_create(int scheme, size_t poly_modulus_degree, const uint64_t *coeff_modulus, size_t k,
                         uint64_t plain_modulus, int device, sb200_context **out);
int sb200_context_destroy(sb200_context *ctx);
/* helpers that reproduce CoeffModulus::Create (modulus.cpp:144-184) */
int sb200_coeff_modulus_create(size_t poly_modulus_degree, const int *bit_sizes, size_t k, uint64_t *out);
/* table introspection for parity tests: NTTTables::get_root / get_from_root_powers / get_from_inv_root_powers /
 * inv_degree_modulo (ntt.h:95-123) in the reference's own order; any output pointer may be NULL */
int sb200_get_ntt_tables(const sb200_context *ctx, size_t prime_index, uint64_t *root, uint64_t *root_powers_operand,
                         uint64_t *root_powers_quotient, uint64_t *inv_root_powers_operand, uint64_t *inv_degree_modulo);
/* RNSTool::base_Bsk() at the level with L primes (rns.h:246-309); out gets |Bsk| values */
int sb200_get_base_bsk(const sb200_context *ctx, size_t L, uint64_t *out, size_t capacity, size_t *count);
/* GaloisTool::get_elt_from_step (galois.cpp:53-95); returns 0 on invalid step */
uint32_t sb200_galois_elt_from_step(const sb200_context *ctx, int step);
/* number of CUDA kernels launched through this context so far */
unsigned long long sb200_launch_count(const sb200_context *ctx);
/* device bytes currently held by the context (tables + scratch) */
size_t sb200_device_bytes(const sb200_context *ctx);
/* resource limits of a context (the reference's counterpart is the MemoryPoolHandle a caller passes to Evaluator members,
 * evaluator.h:219-252): how a batch is cut into device chunks.  Results never depend on them; the parity tests use them
 * to force the multi-chunk paths (ragged last chunk) at small batch sizes.
 *   SB200_LIMIT_SCRATCH_BYTES     budget of the per-context scratch arena (default 8 GiB, env SB200_SCRATCH_MB)
 *   SB200_LIMIT_KS_CHUNK          max ciphertexts per key-switching chunk (0 = derived from the scratch budget)
 *   SB200_LIMIT_HOST_STAGE_BYTES  device staging per pipeline slot of the *_host entry points (default 640 MiB)
 *   SB200_LIMIT_KS_ALGORITHM      key switching: 0 = 64-bit digit transforms per output prime; 1 (default, env SB200_KS_ALGO) =
 *                                 automatic: the exact integer convolution on 29-bit auxiliary primes where it is available
 *                                 (n >= 4096) and pays (levels with >= 6 digits, env SB200_KS_MIN_DIGITS); 2 = that path at every
 *                                 level.  Results are identical words in every mode. */
#define SB200_LIMIT_SCRATCH_BYTES 0
#define SB200_LIMIT_KS_CHUNK 1
#define SB200_LIMIT_HOST_STAGE_BYTES 2
#define SB200_LIMIT_KS_ALGORITHM 3
int sb200_context_set_limit(sb200_context *ctx, int which, size_t value);

/* ---- device-resident slabs (the storage behind seal_b200::CiphertextBatch, include/seal_b200/batch.hpp) ------------
 * The reference hands out ciphertext storage from a MemoryPoolHandle (memorymanager.h:36-54, ciphertext.h:100-140); a
 * caller that keeps ciphertexts on the device between Evaluator calls allocates their slabs here.  Slabs belong to the
 * context's device; sb200_host_malloc returns page-locked host memory (first-touched by the calling thread, so bind the
 * thread to the device's NUMA node first) for staging that the *_host entry points and the copies below can stream
 * from at full PCIe rate.  Copies are stream-ordered; sb200_stream_synchronize(ctx, stream) waits for them. */
int sb200_device_malloc(sb200_context *ctx, size_t bytes, uint64_t **d_out);
int sb200_device_free(sb200_context *ctx, uint64_t *d_ptr);
int sb200_host_malloc(sb200_context *ctx, size_t bytes, void **h_out);
int sb200_host_free(sb200_context *ctx, void *h_ptr);
int sb200_memcpy_h2d(sb200_context *ctx, uint64_t *d_dst, const void *h_src, size_t bytes, void *stream);
int sb200_memcpy_d2h(sb200_context *ctx, void *h_dst, const uint64_t *d_src, size_t bytes, void *stream);
int sb200_memcpy_d2d(sb200_context *ctx, uint64_t *d_dst, const uint64_t *d_src, size_t bytes, void *stream);
/* strided copies between ciphertext objects and slabs: `rows` runs of row_bytes, source / destination pitch in bytes
 * (drops or keeps RNS components without touching the rest: mod_switch_drop_to_next, evaluator.cpp:1296-1358) */
int sb200_memcpy_d2d_2d(sb200_context *ctx, uint64_t *d_dst, size_t dst_pitch, const uint64_t *d_src, size_t src_pitch, size_t row_bytes,
                        size_t rows, void *stream);
int sb200_stream_synchronize(sb200_context *ctx, void *stream);
/* gather / scatter between `count` separate host objects (e.g. seal::Ciphertext::data() of a std::vector<Ciphertext>, pageable
 * pool memory) and one device slab [count][row_bytes]: staged through page-locked double buffers owned by the context, several
 * host threads copy, H2D / D2H overlap the host copies.  Both return when the data has arrived. */
int sb200_upload_rows(sb200_context *ctx, uint64_t *d_dst, const uint64_t *const *h_rows, size_t row_bytes, size_t count);
int sb200_download_rows(sb200_context *ctx, uint64_t *const *h_rows, const uint64_t *d_src, size_t row_bytes, size_t count);
/* NUMA node of the context's device (-1 when the platform does not say) and the CUDA device index */
int sb200_device_numa_node(const sb200_context *ctx);
int sb200_device_index(const sb200_context *ctx);
/* ciphertexts per key-switching chunk the context would use for `batch` ciphertexts at level L (fused != 0: the
 * multiply_relinearize entry point).  bench.py samples its verification indices on both sides of a chunk boundary. */
size_t sb200_keyswitch_chunk(const sb200_context *ctx, size_t L, size_t batch, int fused);

/* ---- per-kernel timing (CUDA events on the launching stream) -------------------------------------------------
 * enable, run operations, then read entries 0,1,... until SB200_E_OUT_OF_RANGE.  Each entry aggregates one kernel
 * (a transform contributes "<name>:col" and "<name>:local"): total device ms, launches, and the algorithmic bytes
 * those launches had to move (DESIGN.md lists the per-kernel formula).  Used by bench.py for the roofline line. */
int sb200_profile_enable(sb200_context *ctx, int on);
int sb200_profile_reset(sb200_context *ctx);
int sb200_profile_read(sb200_context *ctx, size_t index, char *name, size_t name_capacity, double *total_ms,
                       unsigned long long *launches, double *algorithmic_bytes);
/* the same plus the arithmetic those launches executed: modular butterflies and 64x64-bit key multiply-accumulates (per
 * coefficient, not per warp) -- the work of the second ceiling of SURVEY 8(d), the integer-multiply issue rate */
int sb200_profile_read_work(sb200_context *ctx, size_t index, char *name, size_t name_capacity, double *total_ms,
                            unsigned long long *launches, double *algorithmic_bytes, double *butterflies, double *macs);
/* that ceiling, measured in this process on the context's device: the path's own butterfly / multiply-accumulate code on
 * registers only, at the launch shapes of the dominant kernels.  kind 0: forward butterflies (column-pass shape), 1: forward
 * butterflies (fused kernel's shape), 2: inverse butterflies, 3: key multiply-accumulates.  Result: warp-level operations per
 * second of the whole device (one warp-level operation = 32 coefficient-level ones). */
int sb200_selftest_rate(sb200_context *ctx, int kind, double *warp_ops_per_second);
/* the integer key-switching path (SB200_LIMIT_KS_ALGORITHM 1): its work is counted in 32-bit butterflies and 32x32->64-bit
 * multiply-accumulates (sb200_profile_read_work32 = sb200_profile_read_work + those two counters); sb200_selftest_rate kinds
 * 10, 11, 12 measure their ceilings (forward butterflies, inverse butterflies, multiply-accumulates); 13, 14, 15 repeat the
 * multiply-accumulate loop at the key-tile kernel's launch shape (512 threads, one CTA per SM), with two products per accumulator and
 * round (the product kernel's form: one three-input 64-bit add per pair), and with both.  The transforms modulo the
 * auxiliary primes are exposed for the parity tests: _info returns the primes (capacity 8), _forward maps rows of n 64-bit
 * words to h_out[prime][row][n] (canonical residues, transformed), _inverse transforms h_data[row][prime][n] in place (values
 * in [0, 2p), not scaled by n^-1). */
int sb200_profile_read_work32(sb200_context *ctx, size_t index, char *name, size_t name_capacity, double *total_ms,
                              unsigned long long *launches, double *algorithmic_bytes, double *butterflies, double *macs,
                              double *butterflies32, double *macs32);
int sb200_selftest_ksint_info(sb200_context *ctx, int *count, uint32_t *primes);
int sb200_selftest_ksint_forward(sb200_context *ctx, const uint64_t *h_rows, size_t rows, uint32_t *h_out);
int sb200_selftest_ksint_inverse(sb200_context *ctx, uint32_t *h_data, size_t rows);

/* ---- key-switching keys --------------------------------------------------------------------------------------
 * h_key = the flattened KSwitchKeys::data()[index]: [digit j < digits][component 2][key prime k][coeff n], i.e. for
 * each j the PublicKey's ciphertext data (kswitchkeys.h, keygenerator.cpp:327-360).  digits must be >= L of every
 * ciphertext it is used with (evaluator.cpp:2635).  For n >= 4096 the handle also holds the key modulo the context's 29-bit
 * auxiliary primes in transformed form (2.5x the bytes above, prepared once at creation: INTT of every key row + the small
 * forward transforms), which is what key switching at levels with >= 6 digits multiplies with (SB200_LIMIT_KS_ALGORITHM). */
int sb200_kswitch_key_create(sb200_context *ctx, const uint64_t *h_key, size_t digits, sb200_kswitch_key **out);
int sb200_kswitch_key_destroy(sb200_kswitch_key *key);
/* KSwitchKeys::load of the single entry data()[index] out of a RelinKeys / GaloisKeys stream saved with
 * compr_mode_type::none (kswitchkeys.cpp:42-160): the key polynomials go from the stream to the device directly.
 * index = RelinKeys::get_index(2) = 0 for relinearization, GaloisKeys::get_index(galois_elt) = (galois_elt - 1) / 2 for a
 * rotation (relinkeys.h:58-65, galoiskeys.h:48-51).  SB200_E_OUT_OF_RANGE: no such slot; SB200_E_INVALID_ARG: empty slot. */
int sb200_kswitch_key_load(sb200_context *ctx, const uint8_t *stream, size_t len, size_t index, sb200_kswitch_key **out);

/* ---- device-resident batch operations (stream = cudaStream_t, may be NULL) ----------------------------------
 * Output slabs must not alias input slabs unless noted: multiply_relinearize may write over d_a or d_b, add/sub/negate/multiply_plain
 * may run in place; relinearize / rescale / mod_switch / apply_galois change the layout and reject aliasing.
 * The *_host variants stage the batch through the device in chunks (SB200_LIMIT_HOST_STAGE_BYTES; a batch of 4 or more always
 * takes at least two).  When the batch fits one chunk, host output and input buffers may overlap in any way.  With several chunks
 * the output may overlap an input only exactly in place (h_out == that input) with an output no larger than that input, as in
 * add / sub / negate, multiply_plain, relinearize, apply_galois or rescale; any other overlap returns SB200_E_INVALID_ARG before
 * anything is copied. */
/* Evaluator::transform_to_ntt_inplace / transform_from_ntt_inplace (evaluator.cpp:2289-2382) */
int sb200_ntt_forward(sb200_context *ctx, size_t L, size_t size, size_t batch, uint64_t *d_data, void *stream);
int sb200_ntt_inverse(sb200_context *ctx, size_t L, size_t size, size_t batch, uint64_t *d_data, void *stream);
/* Evaluator::multiply (evaluator.cpp:352-708), size-2 x size-2 -> size-3; CKKS (NTT form) or BFV (BEHZ) per ctx */
int sb200_multiply(sb200_context *ctx, size_t L, size_t batch, const uint64_t *d_a, const uint64_t *d_b,
                   uint64_t *d_out3, void *stream);
/* the general-size branches of the same function (evaluator.cpp:524-560, :664-700, :796-833): size_a x size_b ->
 * size_a + size_b - 1, out[k] = sum_{i+j=k} a_i * b_j; 2 <= size <= 16 (SEAL_CIPHERTEXT_SIZE_MAX).  No aliasing. */
int sb200_multiply_sized(sb200_context *ctx, size_t L, size_t size_a, size_t size_b, size_t batch, const uint64_t *d_a,
                         const uint64_t *d_b, uint64_t *d_out, void *stream);
/* Evaluator::square (evaluator.cpp:843-1142): same residues as multiply(a, a), size 2 -> 3 */
int sb200_square(sb200_context *ctx, size_t L, size_t batch, const uint64_t *d_a, uint64_t *d_out3, void *stream);
/* Evaluator::add / sub / negate on equal-size operands (evaluator.cpp:130-350), element-wise over [batch][size][L][n];
 * these are the "next" row of SURVEY 8(f): the linear ops users interleave with multiply / relinearize / rescale */
int sb200_add(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *d_a, const uint64_t *d_b, uint64_t *d_out, void *stream);
int sb200_sub(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *d_a, const uint64_t *d_b, uint64_t *d_out, void *stream);
int sb200_negate(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *d_a, uint64_t *d_out, void *stream);
/* Evaluator::multiply_plain with ciphertext and plaintext both in NTT form (evaluator.cpp:1975-1994 -> multiply_plain_ntt
 * :2157-2195): every polynomial of the ciphertext times the plaintext, dyadic.  d_plain is [batch][L][n]: one NTT-form
 * plaintext per ciphertext, at the ciphertext's level (Plaintext::data() with parms_id == the ciphertext's).  May run in place. */
int sb200_multiply_plain(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *d_a, const uint64_t *d_plain,
                         uint64_t *d_out, void *stream);
/* ---- coefficient-form plaintexts (BFV / BGV): d_plain is [batch][n] words < plain_modulus, zero above coeff_count ----
 * Evaluator::transform_to_ntt_inplace(Plaintext&, parms_id) (evaluator.cpp:2197-2287): lift to the level with L primes
 * (words >= (t+1)/2 are negative, :2240-2272) and transform; d_out is [batch][L][n] */
int sb200_plain_to_ntt(sb200_context *ctx, size_t L, size_t batch, const uint64_t *d_plain, uint64_t *d_out, void *stream);
/* Evaluator::multiply_plain with such a plaintext: multiply_plain_normal (:2021-2155) for coefficient-form ciphertexts
 * (ct_is_ntt = 0, BFV), transform + multiply_plain_ntt (:1999-2004) for NTT-form ciphertexts (BGV).  May run in place. */
int sb200_multiply_plain_coeff(sb200_context *ctx, size_t L, size_t size, size_t batch, int ct_is_ntt, const uint64_t *d_a,
                               const uint64_t *d_plain, uint64_t *d_out, void *stream);
/* Evaluator::add_plain / sub_plain with such a plaintext: BFV adds round(q m / t) to c_0 (util/scalingvariant.cpp:70-160);
 * BGV adds NTT(lift(m * correction_factor mod t)) (:1838-1849), h_correction_factors = [batch] host words or NULL (= 1).
 * May run in place. */
int sb200_add_plain_coeff(sb200_context *ctx, size_t L, size_t size, size_t batch, int subtract, const uint64_t *d_a,
                          const uint64_t *d_plain, const uint64_t *h_correction_factors, uint64_t *d_out, void *stream);
/* BatchEncoder::encode / decode (batchencoder.cpp:84-330; SURVEY 8f rank 4): d_values [batch][n] matrix slots (< t,
 * row-major 2 x n/2) <-> coefficient-form plaintexts d_plain [batch][n].  Needs an NTT-friendly plain modulus
 * (t prime, t = 1 mod 2n: "encryption parameters are not valid for batching" otherwise).  No aliasing. */
int sb200_batch_encode(sb200_context *ctx, size_t batch, const uint64_t *d_values, uint64_t *d_plain, void *stream);
int sb200_batch_decode(sb200_context *ctx, size_t batch, const uint64_t *d_plain, uint64_t *d_values, void *stream);
/* Evaluator::relinearize_inplace, size 3 -> 2 (evaluator.cpp:1144-1199 + 2561-2867) */
int sb200_relinearize(sb200_context *ctx, size_t L, size_t batch, const uint64_t *d_in3,
                      const sb200_kswitch_key *relin_key, uint64_t *d_out2, void *stream);
/* multiply followed by relinearize_inplace in one call; the size-3 intermediate never reaches the caller */
int sb200_multiply_relinearize(sb200_context *ctx, size_t L, size_t batch, const uint64_t *d_a, const uint64_t *d_b,
                               const sb200_kswitch_key *relin_key, uint64_t *d_out2, void *stream);
/* Evaluator::rescale_to_next (CKKS; evaluator.cpp:1503-1541, rns.cpp:830-901): [2][L][n] -> [2][L-1][n] */
int sb200_rescale_to_next(sb200_context *ctx, size_t L, size_t batch, const uint64_t *d_in2, uint64_t *d_out2, void *stream);
/* Evaluator::mod_switch_to_next: BFV divide-and-round (rns.cpp:789-828); CKKS drops the last prime */
int sb200_mod_switch_to_next(sb200_context *ctx, size_t L, size_t batch, const uint64_t *d_in2, uint64_t *d_out2, void *stream);
/* the same two functions for ciphertexts of any size (the reference applies the step to every polynomial, evaluator.cpp:1263-1280):
 * d_in [batch][size][L][n] -> d_out [batch][size][L-1][n] */
int sb200_rescale_to_next_sized(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *d_in, uint64_t *d_out, void *stream);
int sb200_mod_switch_to_next_sized(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *d_in, uint64_t *d_out, void *stream);
/* one step of relinearize_internal's loop (evaluator.cpp:1176-1187) on ciphertexts of size >= 3: d_out = d_in with
 * (c_0, c_1) += switch_key(c_{size-1}, key); every other polynomial is copied, the size is unchanged (the caller drops
 * polynomials when the loop is done, as the reference's final resize does).  No aliasing. */
int sb200_relinearize_sized(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *d_in, const sb200_kswitch_key *key,
                            uint64_t *d_out, void *stream);
/* Evaluator::apply_galois (evaluator.cpp:2384-2502): automorphism x -> x^galois_elt on both polys + key switch.
 * rotate_rows / rotate_vector(step) = apply_galois(sb200_galois_elt_from_step(step)) with that element's key. */
int sb200_apply_galois(sb200_context *ctx, size_t L, size_t batch, const uint64_t *d_in2, uint32_t galois_elt,
                       const sb200_kswitch_key *galois_key, uint64_t *d_out2, void *stream);

/* ---- host-buffer variants: H2D copy, operation, D2H copy, synchronise (the plugin-facing end-to-end path) ---- */
int sb200_ntt_forward_host(sb200_context *ctx, size_t L, size_t size, size_t batch, uint64_t *h_data);
int sb200_ntt_inverse_host(sb200_context *ctx, size_t L, size_t size, size_t batch, uint64_t *h_data);
int sb200_multiply_host(sb200_context *ctx, size_t L, size_t batch, const uint64_t *h_a, const uint64_t *h_b, uint64_t *h_out3);
int sb200_multiply_sized_host(sb200_context *ctx, size_t L, size_t size_a, size_t size_b, size_t batch, const uint64_t *h_a,
                              const uint64_t *h_b, uint64_t *h_out);
int sb200_square_host(sb200_context *ctx, size_t L, size_t batch, const uint64_t *h_a, uint64_t *h_out3);
int sb200_add_host(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *h_a, const uint64_t *h_b, uint64_t *h_out);
int sb200_sub_host(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *h_a, const uint64_t *h_b, uint64_t *h_out);
int sb200_negate_host(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *h_a, uint64_t *h_out);
int sb200_multiply_plain_host(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *h_a, const uint64_t *h_plain,
                              uint64_t *h_out);
int sb200_plain_to_ntt_host(sb200_context *ctx, size_t L, size_t batch, const uint64_t *h_plain, uint64_t *h_out);
int sb200_multiply_plain_coeff_host(sb200_context *ctx, size_t L, size_t size, size_t batch, int ct_is_ntt, const uint64_t *h_a,
                                    const uint64_t *h_plain, uint64_t *h_out);
int sb200_add_plain_coeff_host(sb200_context *ctx, size_t L, size_t size, size_t batch, int subtract, const uint64_t *h_a,
                               const uint64_t *h_plain, const uint64_t *h_correction_factors, uint64_t *h_out);
int sb200_batch_encode_host(sb200_context *ctx, size_t batch, const uint64_t *h_values, uint64_t *h_plain);
int sb200_batch_decode_host(sb200_context *ctx, size_t batch, const uint64_t *h_plain, uint64_t *h_values);
int sb200_relinearize_host(sb200_context *ctx, size_t L, size_t batch, const uint64_t *h_in3,
                           const sb200_kswitch_key *relin_key, uint64_t *h_out2);
int sb200_multiply_relinearize_host(sb200_context *ctx, size_t L, size_t batch, const uint64_t *h_a, const uint64_t *h_b,
                                    const sb200_kswitch_key *relin_key, uint64_t *h_out2);
int sb200_rescale_to_next_host(sb200_context *ctx, size_t L, size_t batch, const uint64_t *h_in2, uint64_t *h_out2);
int sb200_mod_switch_to_next_host(sb200_context *ctx, size_t L, size_t batch, const uint64_t *h_in2, uint64_t *h_out2);
int sb200_apply_galois_host(sb200_context *ctx, size_t L, size_t batch, const uint64_t *h_in2, uint32_t galois_elt,
                            const sb200_kswitch_key *galois_key, uint64_t *h_out2);
int sb200_rescale_to_next_sized_host(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *h_in, uint64_t *h_out);
int sb200_mod_switch_to_next_sized_host(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *h_in, uint64_t *h_out);
int sb200_relinearize_sized_host(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *h_in, const sb200_kswitch_key *key,
                                 uint64_t *h_out);

/* ---- wire format (SURVEY 8f rank 3): Ciphertext::save / load with compr_mode_type::none, straight between a byte
 * stream and a device slab (ciphertext.cpp:190-359, serialization.h:76-91, dynarray.h:662-690).  Seed-compressed ciphertexts
 * (Serializable<Ciphertext> of a symmetric-key encryption: c_1 replaced by the seed of the PRNG that made it) are expanded on
 * the device -- Ciphertext::expand_seed -> sample_poly_uniform on a Blake2xbPRNG (ciphertext.cpp:118-150, util/rlwe.cpp:104-132,
 * randomgen.cpp:204-214), bit for bit -- so a fresh ciphertext crosses PCIe with half its bytes.  zlib-compressed objects
 * (compr_mode_type::zlib, serialization.cpp:236-300, util/ztools.cpp) are inflated on the host with the system's zlib before
 * they are parsed; zstd streams and the shake256 PRNG stay with the reference: load rejects them. */
typedef struct sb200_ct_info
{
    uint64_t parms_id[4];         /* Ciphertext::parms_id() */
    uint64_t size;                /* polynomials */
    uint64_t poly_modulus_degree;
    uint64_t coeff_modulus_size;  /* L */
    uint64_t correction_factor;   /* BGV */
    double scale;                 /* CKKS */
    int32_t is_ntt_form;
    int32_t seeded;               /* 0: both polynomials are stored; otherwise only c_0 is, and c_1 is the output of the PRNG of this
                                     prng_type (randomgen.h:29-36: 1 = blake2xb, 2 = shake256) on the 64-byte seed at seed_offset */
    uint64_t data_offset;         /* byte offset of the first coefficient word in the stream */
    uint64_t data_words;          /* 64-bit words stored */
    uint64_t stream_bytes;        /* length of the serialized object (SEALHeader::size) */
    uint64_t seed_offset;         /* seeded streams: byte offset of the prng_seed_type (64 bytes); 0 otherwise */
    uint64_t compr_mode;          /* compr_mode_type of the stream (serialization.h:33-47): 0 none, 1 zlib; for a compressed stream the
                                     offsets above refer to the decompressed object and stream_bytes to the stream as given */
} sb200_ct_info;

/* EncryptionParameters::parms_id() of the level with L primes (L = k: the key level); encryptionparams.cpp:124-158 */
int sb200_get_parms_id(const sb200_context *ctx, size_t L, uint64_t out[4]);
/* Serialization::LoadHeader + the metadata half of Ciphertext::load_members; pure host, needs no context */
int sb200_ciphertext_inspect(const uint8_t *stream, size_t len, sb200_ct_info *info);
/* bytes Ciphertext::save(compr_mode_type::none) produces for size polynomials at the level with L primes */
size_t sb200_ciphertext_save_size(const sb200_context *ctx, size_t L, size_t size);
/* Ciphertext::load (validate != 0; also checks every residue < q_i like is_data_valid_for, valcheck.cpp) or unsafe_load
 * (validate == 0) of `batch` serialized ciphertexts of one shape into d_out [batch][size][L][n]; infos may be NULL.
 * The coefficient words are copied from the streams to the device directly; seeded streams (size 2) upload c_0 and expand
 * c_1 on the device. */
int sb200_ciphertext_load(sb200_context *ctx, size_t batch, const uint8_t *const *streams, const size_t *lens, size_t L, size_t size,
                          int validate, uint64_t *d_out, sb200_ct_info *infos, void *stream);
/* Ciphertext::save(compr_mode_type::none) of d_in [batch][size][L][n] into outs[b] (capacity >= sb200_ciphertext_save_size);
 * meta[b] supplies is_ntt_form / scale / correction_factor (parms_id, sizes and offsets are filled in here).  Returns after
 * the bytes are in place. */
int sb200_ciphertext_save(sb200_context *ctx, size_t batch, size_t L, size_t size, const uint64_t *d_in, const sb200_ct_info *meta,
                          uint8_t *const *outs, size_t capacity, void *stream);

/* ---- public-key encryption (SURVEY 8f rank 4): Encryptor(context, public_key) and Encryptor::encrypt_zero(parms_id, destination)
 * (encryptor.cpp:88-174 -> util::encrypt_zero_asymmetric, util/rlwe.cpp:184-276) for a batch.
 * h_public_key = PublicKey::data().data(): [2][k][n] words, NTT form at the key level (range-checked).
 * d_out = [batch][2][L][n] at the level with L primes (L == k: the key level): NTT form for CKKS / BGV, coefficient form for BFV,
 * scale 1, correction factor 1.  As in the reference the sample is drawn one level above (L + 1 primes) and divided down by that
 * level's last prime.  Per ciphertext ONE PRNG (Blake2xb of a 64-byte seed) yields the ternary polynomial u and the two noise
 * polynomials exactly as the reference draws them (u through std::uniform_int_distribution as libstdc++ >= 11 implements it),
 * so the same seed gives the reference's ciphertext bit for bit.  h_seeds = [batch][8] words or NULL = fresh seeds from the OS
 * entropy source.  Synchronises the stream.  Add the plaintext as for the symmetric variant to obtain Encryptor::encrypt. */
int sb200_public_key_create(sb200_context *ctx, const uint64_t *h_public_key, sb200_public_key **out);
int sb200_public_key_destroy(sb200_public_key *key);
int sb200_encrypt_zero_asymmetric(sb200_context *ctx, sb200_public_key *key, size_t L, size_t batch, const uint64_t *h_seeds,
                                  uint64_t *d_out, void *stream);

/* ---- CKKSEncoder (SURVEY 8f: the data format either side of the path): CKKSEncoder::encode(values, parms_id, scale, plain) and
 * CKKSEncoder::decode(plain, values) (ckks.h:455-807) for a batch.  values = doubles: [batch][count] complex numbers as (re, im)
 * pairs when is_complex, else [batch][count] reals; count <= n/2, missing slots are zero.  plain = [batch][L][n] NTT form at the
 * level with L primes (Plaintext::data() of each plaintext; its parms_id is sb200_get_parms_id(L), its scale the scale given).
 * Bit-exact with the reference: the double-precision transform performs the reference's operations in the reference's order.
 * Errors as the reference throws them (SB200_E_INVALID_ARG): "scale out of bounds", "values must be finite", "encoded values are
 * too large" (the plaintext buffer is left unspecified), "unsupported scheme" for a non-CKKS context.
 * decode writes [batch][n/2] complex numbers as (re, im) pairs; `scale` is Plaintext::scale().  The encode entry points
 * synchronise the stream once (the magnitude check precedes the reduction). */
int sb200_ckks_encode(sb200_context *ctx, size_t L, size_t batch, const double *d_values, size_t count, int is_complex, double scale,
                      uint64_t *d_plain, void *stream);
int sb200_ckks_decode(sb200_context *ctx, size_t L, size_t batch, const uint64_t *d_plain, double scale, double *d_values, void *stream);
int sb200_ckks_encode_host(sb200_context *ctx, size_t L, size_t batch, const double *h_values, size_t count, int is_complex, double scale,
                           uint64_t *h_plain);
int sb200_ckks_decode_host(sb200_context *ctx, size_t L, size_t batch, const uint64_t *h_plain, double scale, double *h_values);

/* ---- decryption (SURVEY 8f rank 4): Decryptor(context, secret_key) and Decryptor::decrypt (decryptor.cpp:62-197) ------
 * h_secret_key = SecretKey::data().data(): [k][n] words, NTT form at the key level.  Powers of the key for ciphertexts
 * of size > 2 are built on the device on first use (compute_secret_key_array, :199-310). */
int sb200_secret_key_create(sb200_context *ctx, const uint64_t *h_secret_key, sb200_secret_key **out);
int sb200_secret_key_destroy(sb200_secret_key *key);
/* Encryptor::encrypt_zero_symmetric(parms_id, destination) for a batch (encryptor.cpp:168-173 -> util/rlwe.cpp:264-408): fresh
 * encryptions of zero under the secret key at the level with L primes, d_out = [batch][2][L][n] (NTT form for CKKS / BGV,
 * coefficient form for BFV; scale 1, correction factor 1).  Per ciphertext ONE bootstrap PRNG (Blake2xb of a 64-byte seed) yields
 * the public seed c_1 is sampled from and the centred binomial noise, exactly as the reference draws them, so that the same
 * bootstrap seed gives the reference's ciphertext bit for bit.  h_bootstrap_seeds = [batch][8] words, or NULL = fresh seeds from
 * the OS entropy source (what the reference's default UniformRandomGeneratorFactory does, randomgen.cpp:34-50).
 * save_seed != 0 selects the Serializable<Ciphertext> variant (differs for BFV only: which domain c_1 is sampled in);
 * h_public_seeds = NULL or [batch][8]: the seed each c_1 expands from (what a seeded stream carries instead of c_1: send
 * (c_0, seed) over the wire and let the receiver expand, sb200_ciphertext_load).  Add the plaintext (sb200_add for NTT-form CKKS plaintexts, sb200_add_plain_coeff for BFV / BGV)
 * to obtain Encryptor::encrypt_symmetric (encryptor.cpp:199-262). */
int sb200_encrypt_zero_symmetric(sb200_context *ctx, sb200_secret_key *key, size_t L, size_t batch, const uint64_t *h_bootstrap_seeds,
                                 int save_seed, uint64_t *d_out, uint64_t *h_public_seeds, void *stream);
/* d_ct [batch][size][L][n] in the scheme's own form -> d_plain: CKKS [batch][L][n] (NTT form, same level; the caller keeps
 * scale and parms_id); BFV [batch][n] coefficients mod t (dot product + decrypt_scale_and_round, rns.cpp:1133-1191);
 * BGV [batch][n] (dot product, INTT, exact base conversion rns.cpp:466-539, times the inverse of the ciphertext's
 * correction factor: h_correction_factors = [batch] host words or NULL for 1). */
int sb200_decrypt(sb200_context *ctx, sb200_secret_key *key, size_t L, size_t size, size_t batch, const uint64_t *d_ct,
                  const uint64_t *h_correction_factors, uint64_t *d_plain, void *stream);
int sb200_decrypt_host(sb200_context *ctx, sb200_secret_key *key, size_t L, size_t size, size_t batch, const uint64_t *h_ct,
                       const uint64_t *h_correction_factors, uint64_t *h_plain);

/* ---- multi-device dispatch (SURVEY 8e): one context per CUDA device of the box, one host thread per device -----------
 * A batch of independent ciphertexts is cut into contiguous slices, slice i goes to device i through that device's own
 * context (tables and keys replicated, no data-path collective); every call returns when all slices are back in the host
 * buffers.  The reference has no counterpart (it is single-threaded per Evaluator call); this is the C++ side of what
 * bench.py does with one process per GPU.  devices == NULL: every visible device. */
typedef struct sb200_group sb200_group;
typedef struct sb200_group_key sb200_group_key; /* one key-switching key replicated on every device of the group */
int sb200_group_create(int scheme, size_t poly_modulus_degree, const uint64_t *coeff_modulus, size_t k, uint64_t plain_modulus,
                       const int *devices, size_t device_count, sb200_group **out);
int sb200_group_destroy(sb200_group *group);
size_t sb200_group_size(const sb200_group *group);
sb200_context *sb200_group_context(sb200_group *group, size_t i); /* the context of device slot i (owned by the group) */
/* first ciphertext and count of slot i's slice of a batch (the same rule for every call; seal_b200/shard.py mirrors it) */
int sb200_group_slice(const sb200_group *group, size_t batch, size_t i, size_t *first, size_t *count);
int sb200_group_kswitch_key_create(sb200_group *group, const uint64_t *h_key, size_t digits, sb200_group_key **out);
int sb200_group_kswitch_key_destroy(sb200_group_key *key);
int sb200_group_multiply_relinearize_host(sb200_group *group, size_t L, size_t batch, const uint64_t *h_a, const uint64_t *h_b,
                                          const sb200_group_key *relin_key, uint64_t *h_out2);
int sb200_group_relinearize_host(sb200_group *group, size_t L, size_t batch, const uint64_t *h_in3, const sb200_group_key *relin_key,
                                 uint64_t *h_out2);
int sb200_group_apply_galois_host(sb200_group *group, size_t L, size_t batch, const uint64_t *h_in2, uint32_t galois_elt,
                                  const sb200_group_key *galois_key, uint64_t *h_out2);
int sb200_group_multiply_host(sb200_group *group, size_t L, size_t batch, const uint64_t *h_a, const uint64_t *h_b, uint64_t *h_out3);
int sb200_group_rescale_to_next_host(sb200_group *group, size_t L, size_t batch, const uint64_t *h_in2, uint64_t *h_out2);
int sb200_group_mod_switch_to_next_host(sb200_group *group, size_t L, size_t batch, const uint64_t *h_in2, uint64_t *h_out2);
int sb200_group_ntt_forward_host(sb200_group *group, size_t L, size_t size, size_t batch, uint64_t *h_data);
int sb200_group_ntt_inverse_host(sb200_group *group, size_t L, size_t size, size_t batch, uint64_t *h_data);

#ifdef __cplusplus
}
#endif
#endif
