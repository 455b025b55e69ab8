/* accmsm -- C-ABI of the B200-native commitment / MSM hot path for arkworks-rs/accumulation.
 *
 * Drop-in boundary (SURVEY.md 8b): the reference crate forbids `unsafe` (src/lib.rs:24) and never calls
 * an MSM itself; every MSM is reached through ark-poly-commit (`PedersenCommitment::commit`,
 * `InnerProductArgPC::{commit, check_individual_opening_challenges}`), which call
 * `ark_ec::msm::VariableBaseMSM::multi_scalar_mul`.  A Rust `accmsm-sys` crate binds exactly the
 * entry points below (INTEGRATION.md shows the stub) and a `[patch]` of ark-poly-commit routes those
 * bodies here.  Plain pointers and sizes only; no allocation crosses the boundary.
 *
 * Data formats (identical to the ark-ff / ark-ec 0.2 memory images, SURVEY.md App. A.4):
 *   field element : 4 x uint64_t little-endian limbs; "mont" = Fp256 Montgomery image (R = 2^256),
 *                   "canon" = BigInteger256 canonical integer
 *   affine point  : 8 x uint64_t = x[4] || y[4] (Montgomery) + a separate infinity byte; the identity
 *                   is written as (0, 1, infinity = 1) exactly like ark-ec's GroupAffine::zero()
 *   curve id      : 0 = Pallas (coordinates Fp, scalars Fq), 1 = Vesta (coordinates Fq, scalars Fp)
 *   field id      : 0 = Fp (Pallas base), 1 = Fq (Pallas scalar)
 *
 * Every call returns 0 or a negative ACCMSM_E_* code; nothing throws or aborts.  Calls are blocking, with one documented
 * exception: the `*_dev` entry points that take a `stream` argument only ENQUEUE when that argument is not NULL (the caller
 * synchronises its stream).  The ctx has one workspace; work left in flight by such a call is ordered before every later
 * call on any stream by an event, so interleaving streams is safe.  Small host arguments (challenges, randomizers) are
 * copied before the call returns: the caller may reuse its buffers immediately, page-locked or not.
 * There is no CPU fallback: without a CUDA device accmsm_init fails with ACCMSM_E_CUDA.  Two O(1) pieces of field arithmetic
 * run on the calling host thread by design: the affine conversion (one inversion) of the un-normalised sums an entry point
 * returns, and the inverse of an opening round's challenge -- never an MSM, a vector kernel or a point addition.
 * A ctx is bound to one GPU (accmsm_init) or to a group of GPUs of one box (accmsm_init_multi) and serialises its calls
 * internally.  Limits: a registered key has < 2^31 bases, and jobs x windows x n < 2^31 per MSM pass (n < 2^27 at the
 * automatic window sizes).
 */
#ifndef ACCMSM_H
#define ACCMSM_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct accmsm_ctx accmsm_ctx;

enum {
    ACCMSM_OK = 0,
    ACCMSM_E_CUDA = -1,      /* CUDA runtime error (accmsm_last_error has the text) */
    ACCMSM_E_ARG = -2,       /* bad argument (null pointer, bad curve/field id, range) */
    ACCMSM_E_HANDLE = -3,    /* unknown or released bases handle */
    ACCMSM_E_NOMEM = -4      /* device or pinned allocation failed */
};

/* ---- context ------------------------------------------------------------------------------------ */
int  accmsm_init(accmsm_ctx **out, int device);
/* One ctx over the GPUs devices[0 .. n_dev) of this box (SURVEY.md 8b / 8e): one host thread and one stream set per device
 * inside the library.  Every HOST-pointer entry point of this header then spans the devices with no change on the caller's
 * side: accmsm_register_bases cuts the key into contiguous point ranges (one per GPU, at least accmsm_set_min_shard points
 * each), each GPU uploads ITS slice of the caller's scalar / vector buffers over its own PCIe link, runs the whole pipeline
 * on its range and stores one un-normalised 128-byte partial per result into device 0's memory over NVLink (peer store from
 * the last kernel; cudaMemcpyPeer without peer access); device 0 adds them and normalises.  accmsm_ipa_final_key expands
 * h(X) per range with no exchange; accmsm_hp_decide / accmsm_hp_product_poly_comm / accmsm_csr_matvec_commit and the
 * element-wise accmsm_vec_* calls shard by the same index ranges (CSR rows with z replicated).  The accmsm_ipa_open_* calls
 * (begin, begin_combined and begin_shard with log_shards == 0 and no z_scale) shard an opening of 2^k coefficients
 * cyclically over G devices, G the largest power of two <= n_dev and <= 2^k with 2^k / G >= min_shard: device g holds
 * key[g::G] and coeffs[g::G] for the first k - log2 G rounds (one 2 x 128-byte exchange per device per round, combined on
 * device 0), device 0 runs the last log2 G rounds; the proof and eval_out are bit-identical to a single-device session.
 * Smaller openings, and begin_shard with log_shards > 0, run on device 0 over a copy of the whole key assembled by peer
 * copies.  The device-pointer (`*_dev`) entry points need a
 * single-device ctx: accmsm_device_ctx(group, i).  This is what the single-process Rust callers
 * (src/ipa_pc_as/mod.rs:836-845, src/hp_as/mod.rs:910-918, src/r1cs_nark_as/mod.rs:1052-1097) bind. */
int  accmsm_init_multi(accmsm_ctx **out, const int *devices, int n_dev);
int  accmsm_device_count(accmsm_ctx *ctx);
accmsm_ctx *accmsm_device_ctx(accmsm_ctx *ctx, int index);      /* owned by the group; NULL when out of range */
/* keys (vectors, rows) are cut into shards of at least min_points elements; 0 = always use every device.  Default 2^16:
 * below that the fixed tail of an MSM outweighs the split (SURVEY.md App. D.8). */
int  accmsm_set_min_shard(accmsm_ctx *ctx, size_t min_points);
void accmsm_destroy(accmsm_ctx *ctx);
const char *accmsm_strerror(int code);
const char *accmsm_last_error(accmsm_ctx *ctx);
/* Page-locked host buffers for scalars / vectors (optional): every host pointer of this API may be pageable, but
 * H2D then runs at ~16 GB/s instead of the PCIe rate.  Returns NULL on failure. */
void *accmsm_host_alloc(size_t bytes);
void  accmsm_host_free(void *p);
/* tuning knobs (0 = automatic): window bits c for the next MSMs */
int  accmsm_set_window_bits(accmsm_ctx *ctx, int c);
/* IpaPC::open sessions: every `rounds` rounds the key folded by the challenges so far is materialised on the device
 * (one shared-scalar batched MSM over the window table) and the session continues on it, while the key the rounds
 * run on still has >= 2^min_log_n points.  rounds = 0: never (every round runs over the registered key).
 * Defaults 5 and 11 (measured, profiles/r02v_fold_policy.txt: 2^18 -> 2^13 -> 2^8 points).  Results are identical either way.  Replaces the per-round key folding
 * `key_l[i] + key_r[i].mul(xi)` of ark-poly-commit ipa_pc `open` (reached from src/ipa_pc_as/mod.rs:454-462). */
int  accmsm_set_ipa_fold(accmsm_ctx *ctx, int rounds, int min_log_n);
/* number of this library's kernels launched by ctx so far (bench.py reports it as gpu_launches) */
uint64_t accmsm_kernel_launches(accmsm_ctx *ctx);
/* CUDA-event time of the last call's device work, split by stage (ms); names in accmsm_stage_name */
int  accmsm_last_timings(accmsm_ctx *ctx, float *ms_out, int max_stages);
const char *accmsm_stage_name(int stage);

/* ---- commitment keys ------------------------------------------------------------------------------
 * Replaces holding `ck.generators` / `comm_key` on the host: the key is registered once (trim / index
 * time: src/ipa_pc_as/mod.rs:507-513, src/hp_as/mod.rs:640-641) and stays resident in HBM.
 * xy: n x 8 u64.  infinity: n bytes or NULL (generators are never the identity; identity bases are
 * accepted and contribute nothing, like ark-ec's add_assign_mixed). */
int accmsm_register_bases(accmsm_ctx *ctx, int curve, const uint64_t *xy, const uint8_t *infinity,
                          size_t n, uint64_t *handle);
int accmsm_release_bases(accmsm_ctx *ctx, uint64_t handle);
/* Optional, once per key: build the window table 2^(c w) * base_i (w < ceil(256/c), c = window_bits in 4..21,
 * 0 = automatic: 10 / 15 / 17 / 20 for keys below 2^13 / 2^15 / 2^20 / from 2^20 points, measured best)
 * next to the key (ceil(256/c) x 64 B per base).  Commitment keys are fixed from trim / index time on
 * (src/ipa_pc_as/mod.rs:507-513, src/hp_as/mod.rs:640-641), so every later MSM on the handle then uses ONE
 * bucket set: one bucket reduction and no window doublings.  Results are identical with or without it. */
int accmsm_precompute_bases(accmsm_ctx *ctx, uint64_t handle, int window_bits);
/* Seeded synthetic key generated on the device (benchmarks / tests; SURVEY.md 8d): base i of the handle is
 * s * G with G = (-1, 2) and s = the 254-bit SplitMix64 value of (seed, first_index + i), so a GPU can build
 * its own shard of a larger key.  accmsm_download_bases copies registered bases back (x || y Montgomery). */
int accmsm_register_synthetic_bases(accmsm_ctx *ctx, int curve, uint64_t seed, uint64_t first_index,
                                    size_t n, uint64_t *handle);
int accmsm_download_bases(accmsm_ctx *ctx, uint64_t handle, size_t offset, size_t n, uint64_t *xy_out);

/* ark-serialize 0.2 wire format (SURVEY.md 8f rank 4; derives at src/ipa_pc_as/data_structures.rs:55, src/hp_as/data_structures.rs:13):
 * a key as `CanonicalSerialize` writes `Vec<GroupAffine<P>>`, minus the 8-byte length prefix: n x 33 B, each the canonical
 * little-endian x (32 B) + a flag byte (bit 7: y is the larger of (y, -y); bit 6: infinity).  Decompression (one square root
 * per point) runs on the device.  Any invalid encoding fails the call with ACCMSM_E_ARG (ark: SerializationError::InvalidData). */
int accmsm_register_bases_compressed(accmsm_ctx *ctx, int curve, const uint8_t *bytes, size_t n, uint64_t *handle);
int accmsm_serialize_bases(accmsm_ctx *ctx, uint64_t handle, size_t offset, size_t n, uint8_t *out /* n x 33 */);

/* ---- MSM ------------------------------------------------------------------------------------------
 * ark_ec::msm::VariableBaseMSM::multi_scalar_mul(&bases[offset..offset+n], &scalars[..n]) followed by
 * into_affine().  scalars: HOST pointer, n x 4 u64; scalars_montgomery = 1 takes the Fp256 image that
 * PedersenCommitment::commit / cm_commit receive (into_repr() happens on the device), 0 takes
 * BigInteger256.  n = 0 returns the identity.  ark-ec truncates to min(len): the caller passes that. */
int accmsm_msm(accmsm_ctx *ctx, uint64_t handle, size_t offset, size_t n, const uint64_t *scalars,
               int scalars_montgomery, uint64_t out_xy[8], uint8_t *out_inf);
/* The literal ark-ec call for bases that are NOT a registered key: VariableBaseMSM::multi_scalar_mul(&bases, &scalars)
 * + into_affine().  In the reference these are the short linear combinations of commitments
 * (src/hp_as/mod.rs:391-406, src/ipa_pc_as/mod.rs:322-343).  bases_xy: n x 8, infinity: n bytes or NULL. */
int accmsm_msm_oneshot(accmsm_ctx *ctx, int curve, const uint64_t *bases_xy, const uint8_t *infinity,
                       const uint64_t *scalars, int scalars_montgomery, size_t n, uint64_t out_xy[8], uint8_t *out_inf);
/* m such one-shot MSMs of equal length n, each over its own bases, in shared passes of the pipeline (up to 8 per pass): the
 * succinct-check group equations of every input and accumulator of one ipa-pc-as prove / verify (IpaPC::succinct_check is
 * called once per input instance: src/ipa_pc_as/mod.rs:198-205 inside the loops at :262-270 and :625-640; 2k + 3 terms each).
 * bases_xy: m x n x 8, infinity: m x n bytes or NULL, scalars: m x n x 4, out_xy: m x 8, out_inf: m. */
int accmsm_msm_oneshot_batch(accmsm_ctx *ctx, int curve, const uint64_t *bases_xy, const uint8_t *infinity,
                             const uint64_t *scalars, int scalars_montgomery, size_t n, size_t m, uint64_t *out_xy,
                             uint8_t *out_inf);
/* k scalar vectors over the same bases (hp_as::decide commits a, b, a∘b: src/hp_as/mod.rs:910-918;
 * NARK prove commits z_A, z_B, z_C: src/r1cs_nark_as/r1cs_nark/mod.rs:216-218).
 * scalars: k x n x 4 u64, out_xy: k x 8, out_inf: k. */
int accmsm_msm_batch(accmsm_ctx *ctx, uint64_t handle, size_t offset, size_t n, size_t k,
                     const uint64_t *scalars, int scalars_montgomery, uint64_t *out_xy, uint8_t *out_inf);
/* PedersenCommitment::commit(ck, elems, randomizer) / IpaPC::cm_commit(key, scalars, hiding, rand)
 * (SURVEY.md App. A.2): MSM over the first n generators plus randomizer * hiding generator, where the
 * hiding generator is the registered base at index hiding_index.  randomizer_mont may be NULL. */
int accmsm_commit(accmsm_ctx *ctx, uint64_t handle, size_t n, const uint64_t *elems_mont,
                  size_t hiding_index, const uint64_t *randomizer_mont, uint64_t out_xy[8],
                  uint8_t *out_inf);

/* Scalars already resident in HBM (produced on the device by the vector kernels, or staged by the caller):
 * d_scalars is a DEVICE pointer on ctx's GPU; the work is enqueued on `stream` (a cudaStream_t, NULL = the
 * ctx stream) and the call blocks until the affine result is on the host.
 * NOTE for every `stream` argument of this header: the ctx stream is a non-blocking stream and is NOT ordered after
 * work on the CUDA default stream.  A caller whose producer (e.g. an NCCL all-gather issued by torch) runs on the
 * default stream passes that stream explicitly as cudaStreamLegacy ((cudaStream_t)0x1) or cudaStreamPerThread
 * ((cudaStream_t)0x2), never NULL. */
int accmsm_msm_dev(accmsm_ctx *ctx, uint64_t handle, size_t offset, size_t n, const void *d_scalars,
                   int scalars_montgomery, uint64_t out_xy[8], uint8_t *out_inf, void *stream);

/* Device-resident variants for the multi-GPU path (one process per GPU, SURVEY.md 8e): d_scalars is a
 * DEVICE pointer on ctx's GPU, the result is the un-normalised partial sum written to DEVICE memory
 * (16 x u64: X, Y, ZZ, ZZZ), `stream` is a cudaStream_t (NULL = the ctx stream; the call is then
 * synchronous, otherwise it only enqueues). */
int accmsm_msm_partial_dev(accmsm_ctx *ctx, uint64_t handle, size_t offset, size_t n,
                           const void *d_scalars, int scalars_montgomery, void *d_out_partial,
                           void *stream);
/* One GPU's share of accmsm_msm / accmsm_msm_batch / accmsm_commit over a key sharded by point range: k scalar vectors
 * from HOST memory (k x n x 4 u64) against bases [offset, offset + n) of this GPU's handle, optionally a last pair
 * (base tail_index, tail_scalars[j]) per vector (the hiding term of PedersenCommitment::commit, on the shard that owns the
 * hiding generator; tail_scalars in the same representation as scalars, NULL = none).  The k un-normalised sums go to
 * d_out_partials: DEVICE memory, k x 16 u64, possibly on a peer GPU (the final kernel stores there directly).  Blocking. */
int accmsm_msm_partial(accmsm_ctx *ctx, uint64_t handle, size_t offset, size_t n, size_t k, const uint64_t *scalars,
                       int scalars_montgomery, size_t tail_index, const uint64_t *tail_scalars, void *d_out_partials);
/* Sum k gathered partials (DEVICE, k x 16 u64) and normalise: the G-way add after the NCCL gather.
 * Enqueued on `stream` (NULL = the ctx stream); blocks until the affine result is on the host. */
int accmsm_combine_partials_dev(accmsm_ctx *ctx, int curve, const void *d_partials, size_t k,
                                uint64_t out_xy[8], uint8_t *out_inf, void *stream);
/* m results at once: d_partials holds k x m partials, rank-major (exactly what an all-gather of m shares per rank
 * leaves); out_xy m x 8 u64, out_inf m bytes; m <= 8.  Used per round by the multi-GPU IpaPC::open for (l, r). */
int accmsm_combine_partials_batch_dev(accmsm_ctx *ctx, int curve, const void *d_partials, size_t k, size_t m,
                                      uint64_t *out_xy, uint8_t *out_inf, void *stream);

/* ---- IPA decider tail (K3 fused into K2) --------------------------------------------------------------
 * IpaPC::check_individual_opening_challenges after succinct_check (SURVEY.md App. A.2; reached from
 * AtomicASForInnerProductArgPC::decide, src/ipa_pc_as/mod.rs:836-845):
 *   final_key = cm_commit(comm_key, h.compute_coeffs())     with h = SuccinctCheckPolynomial(challenges)
 * The 2^k coefficients are generated on the device inside the digit-decomposition kernel and never
 * touch HBM.  challenges_mont: k x 4 u64, xi_1 first.  The key must hold >= 2^k bases. */
int accmsm_ipa_final_key(accmsm_ctx *ctx, uint64_t handle, const uint64_t *challenges_mont, int k,
                         uint64_t out_xy[8], uint8_t *out_inf);
/* accept iff final_key == proof.final_comm_key (affine equality); *accept = 0/1 */
int accmsm_ipa_check_final_key(accmsm_ctx *ctx, uint64_t handle, const uint64_t *challenges_mont, int k,
                               const uint64_t expected_xy[8], uint8_t expected_inf, int *accept,
                               uint64_t out_xy[8], uint8_t *out_inf);
/* slice [coeff_offset, coeff_offset + n) of the coefficient vector against bases [0, n) of `handle`
 * (a GPU that owns key[coeff_offset ..] registers just that slice); partial stays on the device */
int accmsm_ipa_final_key_partial_dev(accmsm_ctx *ctx, uint64_t handle, const uint64_t *challenges_mont,
                                     int k, size_t coeff_offset, size_t n, void *d_out_partial,
                                     void *stream);

/* ---- IPA opening (IpaPC::open_individual_opening_challenges, SURVEY.md App. A.2) ---------------------------
 * Reference call sites: src/ipa_pc_as/mod.rs:454-462 (AtomicASForInnerProductArgPC::prove), :525-534 (index,
 * default proof), examples/scaling-pc.rs:72-81.  The opening state (coefficients padded to D = 2^k, the
 * z-vector (1, z, z^2, ..), the folded key) lives in HBM for the whole session; the host keeps the sponge:
 *     begin(handle, combined_polynomial_coeffs, k, point, h' = xi_0 * h)
 *     repeat k times:  round() -> (l, r);  xi = sponge(xi_prev, l, r);  fold(xi, xi^-1)
 *     finish() -> (final_comm_key, c)
 * round:  l = cm_commit(key_l, coeffs_r) + <coeffs_r, z_l> h'      r = cm_commit(key_r, coeffs_l) + <coeffs_l, z_r> h'
 * fold :  coeffs_l += xi^-1 coeffs_r;  z_l += xi z_r;  key_l += xi key_r (batch-normalised)
 * fold only enqueues; finish releases the session (also on error).  The key is never folded generator by generator:
 * a round's (l, r) and the final key are MSMs over the registered key (window table if built) with scalars
 * coefficient x product-of-challenges generated in registers, and every few rounds the folded key is materialised in
 * one batched MSM (accmsm_set_ipa_fold) -- results equal the folded-key computation exactly. */
int accmsm_ipa_open_begin(accmsm_ctx *ctx, uint64_t handle, const uint64_t *coeffs_mont, size_t n_coeffs, int k,
                          const uint64_t point_mont[4], const uint64_t h_prime_xy[8], uint64_t *session);
/* Same session, but the polynomial being opened is built on the device: AtomicASForInnerProductArgPC::prove opens
 * the combined succinct-check polynomial P = [random linear poly] + sum_j alpha_j h_j(X) (src/ipa_pc_as/mod.rs:391-404)
 * at the new challenge point; eval_out receives P(point) (:439).  challenges: m x k x 4, xi_1 first. */
int accmsm_ipa_open_begin_combined(accmsm_ctx *ctx, uint64_t handle, const uint64_t *challenges_mont, int m, int k,
                                   const uint64_t *alphas_mont, const uint64_t *random_poly_mont, size_t n_random,
                                   const uint64_t point_mont[4], const uint64_t h_prime_xy[8], uint64_t *session,
                                   uint64_t eval_out[4]);
/* Faster alternative to passing h' as a point: when the hiding generator h is itself a base of the registered key
 * (index h_index) the host passes xi_0 instead (upstream computes h' = ck.h.mul(xi_0)); <., .> h' then rides in each
 * round's MSM as the pair (h, <., .> xi_0) and no separate scalar multiplication happens.  Call after begin (where
 * h_prime_xy may then be NULL) and before the first round. */
int accmsm_ipa_open_use_hiding_generator(accmsm_ctx *ctx, uint64_t session, size_t h_index, const uint64_t xi0_mont[4]);
int accmsm_ipa_open_round(accmsm_ctx *ctx, uint64_t session, uint64_t l_xy[8], uint8_t *l_inf,
                          uint64_t r_xy[8], uint8_t *r_inf);
int accmsm_ipa_open_fold(accmsm_ctx *ctx, uint64_t session, const uint64_t xi_mont[4], const uint64_t xi_inv_mont[4]);
/* One call per round of the loop above: fold with the challenge squeezed from the previous (l, r) -- xi^-1 is computed inside,
 * on the host, like upstream's `round_challenge.inverse()` -- then run the next round; one synchronisation per round.
 * *done = 1 (l, r untouched) when that fold was the last: accmsm_ipa_open_finish follows. */
int accmsm_ipa_open_fold_round(accmsm_ctx *ctx, uint64_t session, const uint64_t xi_mont[4], uint64_t l_xy[8], uint8_t *l_inf,
                               uint64_t r_xy[8], uint8_t *r_inf, int *done);
int accmsm_ipa_open_finish(accmsm_ctx *ctx, uint64_t session, uint64_t final_key_xy[8], uint64_t c_mont[4]);
/* Zero-knowledge opening (MakeZK::Enabled; SURVEY.md 3.2, App. A.2 hiding_comm / rand).  Between begin (or
 * begin_combined) and the first round, in this order:
 *     hide(hiding, s_index, rho) -> hiding_comm;  alpha = sponge(C, z, v, hiding_comm);  hiding_challenge(alpha)
 *     C' = C + alpha hiding_comm - (r + alpha rho) s on the host, xi_0 from C', then the rounds as above
 * hide: uploads the caller's random polynomial (n_hiding <= 2^k coefficients, zero padded), evaluates it at the point and
 *       subtracts the value from coefficient 0 (the polynomial then vanishes there, so eval_out of begin_combined stays
 *       P'(z)), and returns hiding_comm = cm_commit(key[0, 2^k), hiding') + rho key[s_index] from one MSM pass.
 * hiding_challenge: coeffs += alpha hiding' (enqueued only).
 * ACCMSM_E_ARG: hide after the first round or twice, hiding_challenge without hide or twice, a round / fold / finish of a
 * hidden session before its hiding_challenge, n_hiding > 2^k, s_index beyond the key, a session begun with log_shards > 0. */
int accmsm_ipa_open_hide(accmsm_ctx *ctx, uint64_t session, const uint64_t *hiding_coeffs_mont, size_t n_hiding, size_t s_index,
                         const uint64_t hiding_rand_mont[4], uint64_t hiding_comm_xy[8], uint8_t *hiding_comm_inf);
int accmsm_ipa_open_hiding_challenge(accmsm_ctx *ctx, uint64_t session, const uint64_t alpha_mont[4]);

/* Multi-GPU opening (SURVEY.md 8e, "IPA open folding"): the key, the coefficients and the z-vector are sharded
 * CYCLICALLY, shard g of G = 2^log_shards owns the indices i with i mod G == g, so the fold partners i and i + n/2 stay
 * on one GPU until n/2 < G.  Each GPU runs an ordinary session of length 2^k / G over its shard:
 *   begin_shard: z-vector of the shard, z_scale * point^(shard_index + G i); z_scale (nullable = 1) carries the factor
 *                prod_r (1 + xi_r point^(n/2^r)) of rounds folded elsewhere, for the final log2(G) rounds that run
 *                replicated on the G gathered (final key, coefficient) pairs;
 *   round_partial_dev: this shard's un-normalised shares of (l, r) -> 2 x 16 u64 in DEVICE memory (blocking), to be
 *                all-gathered (NCCL) and summed with accmsm_combine_partials_dev; fold / finish as usual.
 * accumulation_b200/sharded.py::ShardedIpaOpen is the host side. */
int accmsm_ipa_open_begin_shard(accmsm_ctx *ctx, uint64_t handle, const uint64_t *coeffs_mont, size_t n_coeffs, int k,
                                const uint64_t point_mont[4], const uint64_t h_prime_xy[8], uint32_t shard_index,
                                uint32_t log_shards, const uint64_t z_scale_mont[4], uint64_t *session);
int accmsm_ipa_open_round_partial_dev(accmsm_ctx *ctx, uint64_t session, void *d_out_partials);

/* ---- field-vector kernels (K3 materialised, K4, K5); all pointers HOST, Montgomery images -------------- */
/* SuccinctCheckPolynomial::compute_coeffs (src/ipa_pc_as/mod.rs:400): out = 2^k elements */
int accmsm_compute_coeffs(accmsm_ctx *ctx, int field, const uint64_t *challenges_mont, int k, uint64_t *out);
/* combine_succinct_check_polynomials (src/ipa_pc_as/mod.rs:391-404):
 * out[j] = random_poly[j] (if j < n_random) + sum_i alphas[i] * coeffs_i[j];  challenges: m x k x 4 */
int accmsm_combine_check_polys(accmsm_ctx *ctx, int field, const uint64_t *challenges_mont, int m, int k,
                               const uint64_t *alphas_mont, const uint64_t *random_poly_mont,
                               size_t n_random, uint64_t *out);
/* DensePolynomial::evaluate (src/ipa_pc_as/mod.rs:439) */
int accmsm_poly_evaluate(accmsm_ctx *ctx, int field, const uint64_t *coeffs_mont, size_t n,
                         const uint64_t *point_mont, uint64_t out[4]);
/* compute_hp (src/hp_as/mod.rs:278-285) */
int accmsm_vec_hadamard(accmsm_ctx *ctx, int field, const uint64_t *a, const uint64_t *b, size_t n, uint64_t *out);
/* scale_vector (src/hp_as/mod.rs:482-489) */
int accmsm_vec_scale(accmsm_ctx *ctx, int field, const uint64_t *v, size_t n, const uint64_t *coeff, uint64_t *out);
/* combine_vectors (src/hp_as/mod.rs:492-512): out[li] = hiding[li] + sum_ni ch[ni] * vecs[ni][li];
 * ragged: vecs[ni] has lens[ni] elements, out has max(lens, n_hiding) elements (out_len receives it) */
int accmsm_vec_lincomb(accmsm_ctx *ctx, int field, const uint64_t *const *vecs, const size_t *lens, int m,
                       const uint64_t *challenges, const uint64_t *hiding, size_t n_hiding,
                       uint64_t *out, size_t out_capacity, size_t *out_len);
/* compute_t_vecs (src/hp_as/mod.rs:288-349): n inputs, mu has n (+1 with hiding) entries,
 * out = (2n-1) x len row-major */
int accmsm_vec_tvecs(accmsm_ctx *ctx, int field, const uint64_t *const *a_vecs, const size_t *a_lens,
                     const uint64_t *const *b_vecs, const size_t *b_lens, int n, const uint64_t *mu,
                     size_t len, const uint64_t *hiding_a, size_t n_ha, const uint64_t *hiding_b,
                     size_t n_hb, uint64_t *out);
/* matrix_vec_mul (src/r1cs_nark_as/r1cs_nark/mod.rs:443-462) for up to 3 CSR matrices sharing z =
 * input || witness in one launch: out[m] = n_rows x 4 u64 */
int accmsm_csr_matvec(accmsm_ctx *ctx, int field, int n_mats, const uint32_t *const *row_ptr,
                      const uint32_t *const *cols, const uint64_t *const *coeffs_mont, size_t n_rows,
                      const uint64_t *input, size_t n_input, const uint64_t *witness, size_t n_witness,
                      uint64_t *const *out);

/* ---- fused steps: vector kernel -> commitments without the vectors leaving HBM (SURVEY.md 8f rank 2) ---------- */
/* ASForHadamardProducts::decide (src/hp_as/mod.rs:894-925): product = a o b; accept iff Commit(a, r1) == comm_1 &&
 * Commit(b, r2) == comm_2 && Commit(product, r3) == comm_3.  The three commitments share one pass of the MSM
 * pipeline.  randomness_mont: 3 x 4 or NULL (no zk); hiding_index: position of the hiding generator in the key. */
int accmsm_hp_decide(accmsm_ctx *ctx, uint64_t handle, const uint64_t *a_mont, const uint64_t *b_mont, size_t n,
                     size_t hiding_index, const uint64_t *randomness_mont, const uint64_t *expected_xy,
                     const uint8_t *expected_inf, int *accept, uint64_t *out_xy, uint8_t *out_inf);
/* One GPU's share of the same decision when the key is sharded by point range (SURVEY.md 8e, K4): a, b are THIS shard's
 * slices (n elements against bases [0, n) of `handle`), the product is formed on the device, and the three un-normalised
 * partial commitments go to d_out_partials (DEVICE memory, 3 x 16 u64, possibly a peer GPU's), to be summed with
 * accmsm_combine_partials_batch_dev.  randomness_mont != NULL only on the shard owning the hiding generator. */
int accmsm_hp_decide_partial_dev(accmsm_ctx *ctx, uint64_t handle, const uint64_t *a_mont, const uint64_t *b_mont, size_t n,
                                 size_t hiding_index, const uint64_t *randomness_mont, void *d_out_partials);
/* compute_t_vecs + compute_product_poly_comm (src/hp_as/mod.rs:288-388): all t-vectors except the middle one are
 * committed (no randomiser).  out_low / out_high: (n_in - 1) x 8; out_tvecs (nullable): (2 n_in - 1) x len x 4. */
int accmsm_hp_product_poly_comm(accmsm_ctx *ctx, uint64_t handle, const uint64_t *const *a_vecs, const size_t *a_lens,
                                const uint64_t *const *b_vecs, const size_t *b_lens, int n_in, const uint64_t *mu,
                                size_t len, const uint64_t *hiding_a, size_t n_ha, const uint64_t *hiding_b, size_t n_hb,
                                uint64_t *out_low_xy, uint8_t *out_low_inf, uint64_t *out_high_xy, uint8_t *out_high_inf,
                                uint64_t *out_tvecs);
/* sharded form: the vectors are this shard's slices; 2 n_in - 2 partials (low rows, then high) -> d_out_partials (DEVICE);
 * row r of the t-vectors (nullable) is written at out_tvecs + r * tvec_row_stride * 4 */
int accmsm_hp_product_poly_comm_partial_dev(accmsm_ctx *ctx, uint64_t handle, const uint64_t *const *a_vecs, const size_t *a_lens,
                                            const uint64_t *const *b_vecs, const size_t *b_lens, int n_in, const uint64_t *mu,
                                            size_t len, const uint64_t *hiding_a, size_t n_ha, const uint64_t *hiding_b, size_t n_hb,
                                            void *d_out_partials, uint64_t *out_tvecs, size_t tvec_row_stride);
/* R1CS matrices registered once (fixed from index time on: src/r1cs_nark_as/r1cs_nark/mod.rs:78-124); then
 * t_M = M (input || witness) and comm_M = Commit(t_M, blinder_M) for all matrices in one call
 * (prover :183-185 + :216-218, verifier :356-361 + :375-389, AS decider src/r1cs_nark_as/mod.rs:1052-1097).
 * out_vecs: NULL or n_mats pointers (each nullable) receiving t_M; blinders_mont: n_mats x 4 or NULL. */
int accmsm_register_csr(accmsm_ctx *ctx, int field, int n_mats, const uint32_t *const *row_ptr, const uint32_t *const *cols,
                        const uint64_t *const *coeffs_mont, size_t n_rows, uint64_t *handle);
int accmsm_release_csr(accmsm_ctx *ctx, uint64_t handle);
int accmsm_csr_matvec_commit(accmsm_ctx *ctx, uint64_t key_handle, uint64_t csr_handle, const uint64_t *input, size_t n_input,
                             const uint64_t *witness, size_t n_witness, size_t hiding_index, const uint64_t *blinders_mont,
                             uint64_t *const *out_vecs, uint64_t *out_xy, uint8_t *out_inf);

/* One GPU's share of the same step when the key -- and with it the rows of the matrices -- is sharded by point range
 * (SURVEY.md 8e, K5): csr_handle holds THIS shard's rows, z = input || witness is replicated, the n_mats un-normalised partial
 * commitments go to d_out_partials (DEVICE memory, possibly a peer GPU's); blinders_mont != NULL only on the shard that owns
 * the hiding generator; out_vecs[m] receive this shard's rows of t_M. */
int accmsm_csr_matvec_commit_partial_dev(accmsm_ctx *ctx, uint64_t key_handle, uint64_t csr_handle, const uint64_t *input, size_t n_input,
                                         const uint64_t *witness, size_t n_witness, size_t hiding_index, const uint64_t *blinders_mont,
                                         uint64_t *const *out_vecs, void *d_out_partials);

/* zk R1CSNark::prove first message (src/r1cs_nark_as/r1cs_nark/mod.rs:183-261): z_M = M (x||w), r_M = M (0||r),
 * cross = z_A o r_B + z_B o r_A, rr = r_A o r_B, and the 8 commitments in ONE pass.  csr_handle must hold 3 matrices.
 * r: n_witness x 4.  blinders: 8 x 4, in the order A, B, C, rA, rB, rC, 1, 2 (required).
 * out_xy: 8 x 8, out_inf: 8, in the same order.  out_vecs: NULL, or 8 nullable pointers (n_rows x 4).
 * The prover then squeezes gamma and forms w' = w + gamma r with accmsm_vec_lincomb (hiding = w, vecs = [r], ch = [gamma]),
 * sigma_M = blinder_M + gamma rblinder_M and sigma_o = blinder_C + gamma blinder_1 + gamma^2 blinder_2 (:262-316).
 * One pass of 8 jobs over n_rows + 1 pairs needs 8 x windows x (n_rows + 1) < 2^31: n_rows < ~2^24 at c = 20.
 * The non-zk prove is accmsm_csr_matvec_commit. */
int accmsm_nark_prove_zk(accmsm_ctx *ctx, uint64_t key_handle, uint64_t csr_handle, const uint64_t *input, size_t n_input,
                         const uint64_t *witness, size_t n_witness, const uint64_t *r, size_t hiding_index,
                         const uint64_t *blinders_mont, uint64_t *const *out_vecs, uint64_t *out_xy, uint8_t *out_inf);
/* R1CSNark::verify (:335-419): t_M = M (x||w'), then Commit(t_A, s_A), Commit(t_B, s_B), Commit(t_C, s_C) and
 * Commit(t_A o t_B, s_o) in ONE pass, compared with expected_xy / expected_inf (4 points, which the caller combines from the
 * proof: comm_M + gamma comm_rM and comm_C + gamma comm_1 + gamma^2 comm_2; without zk comm_A, comm_B, comm_C, comm_C).
 * sigmas: 4 x 4, or NULL without zk.  out_vecs: NULL, or 3 nullable pointers (t_A, t_B, t_C; t_A and t_B are also the
 * hp witnesses of ASForR1CSNark::compute_hp_input_witnesses, src/r1cs_nark_as/mod.rs).  out_xy / out_inf nullable.
 * One pass of 4 jobs: n_rows < ~2^25 at c = 20. */
int accmsm_nark_verify(accmsm_ctx *ctx, uint64_t key_handle, uint64_t csr_handle, const uint64_t *input, size_t n_input,
                       const uint64_t *blinded_witness, size_t n_witness, size_t hiding_index, const uint64_t *sigmas_mont,
                       const uint64_t *expected_xy, const uint8_t *expected_inf, int *accept, uint64_t *out_xy,
                       uint8_t *out_inf, uint64_t *const *out_vecs);
/* ASForR1CSNark::decide (src/r1cs_nark_as/mod.rs:1031-1112): t_M = M (x*||w*) for the 3 matrices of csr_handle, then
 * Commit(t_M, sigma_M*) for M = A, B, C, and the hp decider's Commit(a*, r1*), Commit(b*, r2*), Commit(a* o b*, r3*)
 * (src/hp_as/mod.rs:894-925), all six in ONE pass; accept iff they equal expected_xy / expected_inf in the order
 * comm_A*, comm_B*, comm_C*, C1*, C2*, C3* (out_xy / out_inf, nullable, in the same order).
 * hp_a, hp_b: a* and b* with n_a, n_b <= n_rows (else ACCMSM_E_ARG); the product runs over min(n_a, n_b).
 * sigmas: (sigma_A*, sigma_B*, sigma_C*), hp_rand: (r1*, r2*, r3*), each 3 x 4 or NULL; an absent triple adds nothing.
 * One pass of 6 jobs over n_rows + 1 pairs needs 6 x windows x (n_rows + 1) < 2^31: n_rows <= 27,531,840 (~2^24.7) at c = 20. */
int accmsm_nark_as_decide(accmsm_ctx *ctx, uint64_t key_handle, uint64_t csr_handle, const uint64_t *input, size_t n_input,
                          const uint64_t *witness, size_t n_witness, const uint64_t *hp_a, size_t n_a, const uint64_t *hp_b, size_t n_b,
                          size_t hiding_index, const uint64_t *sigmas_mont, const uint64_t *hp_rand_mont, const uint64_t *expected_xy,
                          const uint8_t *expected_inf, int *accept, uint64_t *out_xy, uint8_t *out_inf);

/* ---- ASForHadamardProducts::prove as a session (src/hp_as/mod.rs:646-813; SURVEY.md App. C.1-C.6) -------------------------
 * The n_in pairs (a_i, b_i) -- inputs first, then old accumulators, after the caller's placeholder padding -- are uploaded
 * once and stay in HBM until finish; the host keeps the sponge and the O(n) pieces (r1*, r2*, r3*, C1*, C2*, C3*):
 *     begin(pairs, hiding) -> hiding comms;  mu = sponge(.., hiding comms)
 *     product_poly_comm(mu) -> low, high;    nu = sponge(.., low, high)
 *     finish(nu) -> a*, b*
 * begin: each a_i, b_i holds a_lens[i] / b_lens[i] <= len elements, len <= the key length.  Zero knowledge: hiding_a and
 *   hiding_b (len x 4 each, both or neither), hiding_rand (r1, r2, r3: 3 x 4) and the generator index hiding_index; begin then
 *   returns Commit(ha, r1), Commit(hb, r2), Commit(ha o b_0 + a_{n-1} o hb, r3) (3 x 8, 3) from one pass.  The last vector is
 *   the hiding part of the middle t-vector, which holds only for n_in >= 2 (with n_in = 1 it also carries mu_1^2 ha o hb):
 *   hiding with n_in = 1 is ACCMSM_E_ARG (the reference's zk padding keeps n >= 2).  Without hiding begin runs no kernel.
 * product_poly_comm: mu = (mu_0 = 1, mu_1 .. mu_{n-1}) and, with hiding, mu_n = mu_1 mu_{n-1} (n_mu = n_in (+1)); low / high:
 *   (n_in - 1) x 8 and n_in - 1 flags each, as accmsm_hp_product_poly_comm.
 * finish: a* = mu_n ha + sum_i mu_i nu^i a_i and b* = mu_1 hb + sum_j nu^j b_{n-1-j} (App. C.5) into a_star / b_star (capacity
 *   elements each); out_len[0] / out_len[1] receive their lengths, max(a_lens (, len with hiding)) and max(b_lens (, len)).
 *   finish releases the session, on error too; abort releases it without results.
 * ACCMSM_E_ARG (the session stays usable unless finish was called): steps out of order, a wrong n_mu, n_in outside
 * 1..16, one hiding vector without the other, hiding with n_in = 1, a vector longer than len.  An unknown session:
 * ACCMSM_E_HANDLE.  Calls on the same ctx between the steps do not disturb a session, and several sessions may be live. */
int accmsm_hp_prove_begin(accmsm_ctx *ctx, uint64_t key_handle, const uint64_t *const *a_vecs, const size_t *a_lens,
                          const uint64_t *const *b_vecs, const size_t *b_lens, int n_in, size_t len, const uint64_t *hiding_a,
                          const uint64_t *hiding_b, size_t hiding_index, const uint64_t *hiding_rand_mont, uint64_t *hiding_comm_xy,
                          uint8_t *hiding_comm_inf, uint64_t *session);
int accmsm_hp_prove_product_poly_comm(accmsm_ctx *ctx, uint64_t session, const uint64_t *mu_mont, size_t n_mu, uint64_t *low_xy,
                                      uint8_t *low_inf, uint64_t *high_xy, uint8_t *high_inf);
int accmsm_hp_prove_finish(accmsm_ctx *ctx, uint64_t session, const uint64_t nu_mont[4], uint64_t *a_star, uint64_t *b_star,
                           size_t capacity, size_t *out_len);
int accmsm_hp_prove_abort(accmsm_ctx *ctx, uint64_t session);

#ifdef __cplusplus
}
#endif
#endif
