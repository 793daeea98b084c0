/* vrfs_b200 - C ABI of the B200 batched VRF engine.
 *
 * This is the drop-in boundary for the data-parallel hot path of `ark-ec-vrfs` (= `ark-vrf` 0.1.0, the
 * sole dependency at /root/reference/Cargo.toml:12).  The reference has no FFI of its own: its boundary
 * is the Rust trait API whose names are re-exported at /root/reference/src/lib.rs:13-17
 * (`Suite, Secret, Public, Input, Output, ietf, pedersen, ring, codec, utils`).  Each entry point below
 * is the BATCH form of one of those items; the Rust shim that keeps the crate's per-item API on top of
 * it is shown in INTEGRATION.md.  Behaviour is specified in SURVEY.md Appendix A.
 *
 * Conventions (all entry points):
 *   - scalars (`Secret`, proof `c`, `s`, `sb`, blinding): 32 bytes little-endian; values >= r are
 *     reduced mod r on load, like `ScalarField::from_le_bytes_mod_order`.  For the SEC1 suite the wire
 *     encoding is big-endian; the ABI is little-endian for every suite.
 *   - points (`Public`, `Input`, `Output`, proof points): affine x || y, 32 bytes little-endian each,
 *     canonical (< p).  Non-canonical or off-curve points make that item fail (out_ok = 0 / zeroed
 *     output); the call itself still returns VRFS_OK.  Points must lie in the prime-order subgroup,
 *     which the reference's typed values guarantee (arkworks validates on deserialisation); the
 *     short-Weierstrass identity is 64 zero bytes.
 *   - variable-length data (`ad`, h2c `data`, seeds): one concatenated byte buffer + n+1 offsets
 *     (uint64).  A NULL `ad` means every item has empty additional data.
 *   - BLS12-381 G1 points: affine x || y, 48 bytes little-endian each; identity = 96 zero bytes.
 *   - Secrets: device staging buffers that held `Secret` scalars, nonces or blinding factors are zeroed before the call
 *     returns (the buffers are pooled, so that is their "release"); the library keeps no pinned host copies.
 *   - The caller owns every buffer; nothing is retained after return.  No exceptions, no aborts:
 *     every failure is a status code; `vrfs_last_error` gives text.  There is NO CPU fallback: without
 *     a CUDA device every call fails with VRFS_CUDA_ERROR.
 *   - `vrfs_*_batch`      : HOST buffers; copies in, runs, copies out, returns when done.
 *     `vrfs_*_batch_dev`  : DEVICE buffers (16-byte aligned) of the same layout, enqueued on the
 *                           context's stream; results are ready after `vrfs_ctx_sync`.
 *   - One context per GPU (one process per GPU under torch.distributed / NCCL).  A context is internally synchronised:
 *     concurrent calls on one context from several host threads serialise (per-context mutex); `*_batch_dev` calls
 *     are asynchronous on the context's stream and must be followed by `vrfs_ctx_sync` before their buffers are reused.
 */
#ifndef VRFS_B200_H
#define VRFS_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct vrfs_ctx vrfs_ctx;
typedef enum { VRFS_OK = 0, VRFS_INVALID_DATA = 1, VRFS_CUDA_ERROR = 2, VRFS_BAD_ARG = 3, VRFS_UNSUPPORTED = 4 } vrfs_status;
/* `suites::{bandersnatch, ed25519, secp256r1}` (lib.rs:13-17; SURVEY A.1) and, per SURVEY 8(f)4, the remaining suites of the crate:
 * bandersnatch_sw ("Bandersnatch_SW_SHA-512_TAI", the short-Weierstrass form; encoded points are arkworks' 33-byte x || flags),
 * jubjub ("JubJub_SHA-512_TAI") and baby-jubjub ("BabyJubJub_SHA-512_TAI").  The last three are PARITY UNPINNED: curve constants are
 * checked numerically, suite strings / CHALLENGE_LEN = 32 are recalled, and their Pedersen blinding bases are placeholders
 * (data_to_point of a fixed label) until the crate's constants are available. */
typedef enum { VRFS_BANDERSNATCH_ELL2 = 0, VRFS_ED25519_TAI = 1, VRFS_P256_TAI = 2, VRFS_BANDERSNATCH_SW_TAI = 3, VRFS_JUBJUB_TAI = 4,
               VRFS_BABYJUBJUB_TAI = 5, VRFS_SUITE_COUNT = 6 } vrfs_suite;
/* Per-item result of the verifiers: the reference's `Result<(), Error>` with `Error::{VerificationFailure, InvalidData}`
 * (/root/reference/src/lib.rs:13-17, `Error`).  Every verify entry point takes an optional `out_status` array (may be NULL)
 * next to `out_ok`:
 *   VRFS_ITEM_OK                    Ok(())                       (out_ok = 1)
 *   VRFS_ITEM_VERIFICATION_FAILURE  well-formed values whose proof does not check
 *   VRFS_ITEM_INVALID_DATA          a value no typed Public / Input / Output / Proof can hold: non-canonical coordinates or
 *                                   scalars, off the curve, the un-encodable short-Weierstrass identity; on the wire entry
 *                                   points also: outside the prime-order subgroup, s >= r, no input point found */
typedef enum { VRFS_ITEM_OK = 0, VRFS_ITEM_VERIFICATION_FAILURE = 1, VRFS_ITEM_INVALID_DATA = 2 } vrfs_item_status;

int vrfs_abi_version(void);
/* device = CUDA ordinal.  The fixed-base tables for G and the Pedersen blinding base B (2 x 50 MB per suite) are built the
 * first time a suite is used, not here. */
vrfs_status vrfs_ctx_create(int device, vrfs_ctx** out);
void vrfs_ctx_destroy(vrfs_ctx* ctx);
vrfs_status vrfs_ctx_sync(vrfs_ctx* ctx);
const char* vrfs_last_error(const vrfs_ctx* ctx);
/* the CUDA stream (cudaStream_t) the context enqueues on; lets a caller order its own work after it */
void* vrfs_ctx_stream(vrfs_ctx* ctx);
/* Page-locked host memory.  Every batch call copies straight from / into the caller's buffers; with page-locked buffers those
 * copies run beside the kernels (all but the first ~20 MB of a 2^20-item call's inputs hide behind arithmetic), with pageable ones
 * the driver stages them synchronously (measured: 12.5 vs ~11 M verifies/s end to end).  vrfs_host_alloc / vrfs_host_free give such
 * memory to callers without a CUDA runtime of their own; vrfs_host_register / vrfs_host_unregister page-lock an existing
 * allocation (e.g. a Rust Vec<u8> that lives across calls) in place.  No context is involved; status only, no message. */
vrfs_status vrfs_host_alloc(size_t bytes, void** out);
vrfs_status vrfs_host_free(void* p);
vrfs_status vrfs_host_register(void* p, size_t bytes);
vrfs_status vrfs_host_unregister(void* p);
/* test hook: n bytes at `offset` of internal staging buffer `slot` (0..4 = the input staging buffers in argument order, e.g.
 * slot 0 held `sk` during a prove call); lets tests check that key material is zeroed once a call has returned */
vrfs_status vrfs_ctx_debug_read_staging(vrfs_ctx* ctx, int slot, size_t offset, uint8_t* out, size_t n);
/* number of kernel launches issued by this context so far (bench.py's `gpu_launches`) */
uint64_t vrfs_ctx_launch_count(const vrfs_ctx* ctx);
/* per-kernel device times (CUDA events on the context's stream) of the most recent batch call; used by
 * bench.py for the roofline of the dominant kernel.  names[i] are static strings. */
vrfs_status vrfs_ctx_enable_kernel_timing(vrfs_ctx* ctx, int on);
int vrfs_ctx_kernel_timings(vrfs_ctx* ctx, const char** names, float* ms, int cap);
/* suite constants: SUITE_ID-independent sizes used by callers to size buffers */
int vrfs_suite_challenge_len(vrfs_suite s);   /* Suite::CHALLENGE_LEN */
int vrfs_suite_hash_len(vrfs_suite s);        /* HashOutput<S> length */
int vrfs_suite_point_enc_len(vrfs_suite s);   /* Codec::point_encode length */

/* Secret::from_seed + Public (lib.rs:13-17; A.3): sk = LE(H(seed)) mod r, pk = sk*G.  out_pk may be NULL. */
vrfs_status vrfs_secret_from_seed_batch(vrfs_ctx*, vrfs_suite, size_t n, const uint8_t* seeds, const uint64_t* seed_off,
                                        uint8_t* out_sk /*n*32*/, uint8_t* out_pk /*n*64*/);
/* Input::new -> Suite::data_to_point (A.5).  out_ok[i] = 0 if no point was found. */
vrfs_status vrfs_data_to_point_batch(vrfs_ctx*, vrfs_suite, size_t n, const uint8_t* data, const uint64_t* data_off,
                                     uint8_t* out_pts /*n*64*/, uint8_t* out_ok /*n*/);
/* Secret::output: O = sk * I */
vrfs_status vrfs_output_batch(vrfs_ctx*, vrfs_suite, size_t n, const uint8_t* sk, const uint8_t* input, uint8_t* out_output /*n*64*/);
/* Output::hash -> Suite::point_to_hash (A.8) */
vrfs_status vrfs_point_to_hash_batch(vrfs_ctx*, vrfs_suite, size_t n, const uint8_t* pts, uint8_t* out_hash /*n*hash_len*/);
/* codec::point_encode / point_decode (A.2) */
vrfs_status vrfs_point_encode_batch(vrfs_ctx*, vrfs_suite, size_t n, const uint8_t* pts, uint8_t* out_enc /*n*enc_len*/);
vrfs_status vrfs_point_decode_batch(vrfs_ctx*, vrfs_suite, size_t n, const uint8_t* enc, uint8_t* out_pts /*n*64*/, uint8_t* out_ok);
/* Suite::nonce (A.6) */
vrfs_status vrfs_nonce_batch(vrfs_ctx*, vrfs_suite, size_t n, const uint8_t* sk, const uint8_t* input, uint8_t* out_k /*n*32*/);

/* ietf::Prover::prove (A.9).  out_c, out_s: n*32 (c is a full 32-byte LE scalar whose value fits cLen bytes). */
vrfs_status vrfs_ietf_prove_batch(vrfs_ctx*, vrfs_suite, size_t n, const uint8_t* sk, const uint8_t* input, const uint8_t* output,
                                  const uint8_t* ad, const uint64_t* ad_off, uint8_t* out_c, uint8_t* out_s);
/* ietf::Verifier::verify (A.9) - the headline metric.  out_ok[i] = 1 iff the proof verifies (Ok(())),
 * 0 for Error::VerificationFailure / Error::InvalidData. */
vrfs_status vrfs_ietf_verify_batch(vrfs_ctx*, vrfs_suite, size_t n, const uint8_t* pk, const uint8_t* input, const uint8_t* output,
                                   const uint8_t* c, const uint8_t* s, const uint8_t* ad, const uint64_t* ad_off, uint8_t* out_ok,
                                   uint8_t* out_status /* n x vrfs_item_status, may be NULL */);
vrfs_status vrfs_ietf_verify_batch_dev(vrfs_ctx*, vrfs_suite, size_t n, const uint8_t* d_pk, const uint8_t* d_input,
                                       const uint8_t* d_output, const uint8_t* d_c, const uint8_t* d_s, const uint8_t* d_ad,
                                       const uint64_t* d_ad_off, uint8_t* d_out_ok, uint8_t* d_out_status /* may be NULL */);

/* ietf::Verifier::verify against PREPARED public keys: "prepare once, verify many" for a known signer set (a validator set, a
 * committee).  vrfs_public_keys_prepare builds, on this context's GPU, one fixed-base table per key (8-bit signed windows, about
 * 400 KB per key), so that c*Y costs 32 mixed additions (16-17 for a 16-byte challenge) instead of a variable-base multiplication.
 *   prepare: n_keys affine keys (x || y, the layout of every typed call) of one suite.  out_key_ok (may be NULL): 1 per key that
 *            vrfs_ietf_verify_batch would accept as a key (canonical, on the curve, not the short-Weierstrass identity), else 0.
 *            1 <= n_keys <= 65536, else VRFS_BAD_ARG.  An allocation that fails returns VRFS_CUDA_ERROR and leaks nothing.
 *   verify:  item i is ietf::Verifier::verify with pk[i] = pks[key_index[i]]: out_ok / out_status are exactly those of
 *            vrfs_ietf_verify_batch on the gathered keys.  key_index[i] >= n_keys makes item i VRFS_ITEM_INVALID_DATA (never an
 *            out-of-range read).  4 bytes of key index travel per item instead of 64 bytes of key.  The _dev form takes 16-byte
 *            aligned device buffers and is asynchronous on the context's stream, like vrfs_ietf_verify_batch_dev.
 * A handle belongs to the context that prepared it; with any other context the calls return VRFS_BAD_ARG.  vrfs_ctx_destroy frees
 * the tables of the handles still alive and orphans them; releasing an orphan (or NULL) only frees its record.
 * Keys are meant to be typed `Public` values, i.e. in the prime-order subgroup (decode them with vrfs_point_decode_checked_batch).
 * For an on-curve key with a small-order component the two calls need not agree on a crafted proof: vrfs_ietf_verify_batch
 * computes c*Y for Bandersnatch through the GLV split k1*Y + k2*psi(Y), which equals c*Y only on the subgroup, while the table
 * computes c*Y itself.  Both reject honest proofs under such a key (its encoding enters the challenge). */
typedef struct vrfs_public_keys vrfs_public_keys;
vrfs_status vrfs_public_keys_prepare(vrfs_ctx*, vrfs_suite, size_t n_keys, const uint8_t* pks /*n_keys*64*/,
                                     uint8_t* out_key_ok /*n_keys, may be NULL*/, vrfs_public_keys** out);
void vrfs_public_keys_release(vrfs_public_keys*);
vrfs_status vrfs_ietf_verify_prepared_batch(vrfs_ctx*, const vrfs_public_keys*, size_t n, const uint32_t* key_index,
                                            const uint8_t* input, const uint8_t* output, const uint8_t* c, const uint8_t* s,
                                            const uint8_t* ad, const uint64_t* ad_off, uint8_t* out_ok, uint8_t* out_status /* may be NULL */);
vrfs_status vrfs_ietf_verify_prepared_batch_dev(vrfs_ctx*, const vrfs_public_keys*, size_t n, const uint32_t* d_key_index,
                                                const uint8_t* d_input, const uint8_t* d_output, const uint8_t* d_c, const uint8_t* d_s,
                                                const uint8_t* d_ad, const uint64_t* d_ad_off, uint8_t* d_out_ok, uint8_t* d_out_status /* may be NULL */);
/* The same from bytes: a signer set published as encoded keys, signatures verified by key index (a block header's author index and
 * seal).  vrfs_public_keys_prepare_encoded decodes each key once like vrfs_point_decode_checked_batch (canonical, on the curve,
 * prime-order subgroup) and prepares the decoded points: out_key_ok[k] = 1 iff the encoding decodes AND vrfs_public_keys_prepare
 * would accept the decoded point.  Such a handle also serves vrfs_ietf_verify_prepared_batch[_dev], exactly like an affine handle
 * of the decoded points, and no key of it has a small-order component, so the caveat above cannot arise.
 * vrfs_ietf_verify_prepared_wire_batch: item i is vrfs_ietf_verify_wire_batch with pk_enc[i] = the encoding of key key_index[i] as
 * given to prepare: out_ok, out_hash and out_status equal that call's byte for byte, for every key encoding.  An item that names a
 * key with key_ok = 0, or an index >= n_keys, is VRFS_ITEM_INVALID_DATA with ok 0 and a zero hash.  Each key is decoded and
 * subgroup-checked once at prepare instead of once per item, 4 bytes of key index travel instead of an encoded key, and
 * U = s*G - c*Y comes from the key's table.  A handle made by vrfs_public_keys_prepare (keys never subgroup-checked) is refused with
 * VRFS_BAD_ARG.  Handle rules, n_keys range and NULL buffers as above; out_hash may be NULL.  There is no _dev form. */
vrfs_status vrfs_public_keys_prepare_encoded(vrfs_ctx*, vrfs_suite, size_t n_keys, const uint8_t* pk_enc /*n_keys*enc_len*/,
                                             uint8_t* out_key_ok /*n_keys, may be NULL*/, vrfs_public_keys** out);
vrfs_status vrfs_ietf_verify_prepared_wire_batch(vrfs_ctx*, const vrfs_public_keys*, size_t n, const uint32_t* key_index,
                                                 const uint8_t* data, const uint64_t* data_off, const uint8_t* sig /*n*sig_len*/,
                                                 const uint8_t* ad, const uint64_t* ad_off,
                                                 uint8_t* out_ok, uint8_t* out_hash /*n*hash_len, may be NULL*/, uint8_t* out_status /* may be NULL */);
/* The same against PREPARED VRF INPUTS: a lottery or beacon round has every participant evaluate the VRF on the round's input, so a
 * batch holds few distinct inputs (JAM/Safrole seals: hundreds of signatures over one to three inputs per epoch).
 * vrfs_inputs_prepare runs Input::new on n_inputs data items once: out_input_ok[j] is the flag of vrfs_data_to_point_batch
 * (0 = no point found) and out_points its points byte for byte; then it builds one table per input point, of the layout and size
 * of a prepared key, so that s*I costs 32-33 mixed additions and V = s*I - c*O keeps one variable base, c*O.
 * 1 <= n_inputs <= 65536, else VRFS_BAD_ARG.
 *   vrfs_ietf_verify_prepared_io_batch[_dev]: item i is vrfs_ietf_verify_prepared_batch with input[i] = points[input_index[i]]
 *     (ok and status), 136 bytes per item instead of 196.  input_index[i] >= n_inputs, or an input with input_ok = 0, makes item
 *     i VRFS_ITEM_INVALID_DATA (never an out-of-range read).  The _dev form takes 16-byte aligned device buffers and is
 *     asynchronous on the context's stream.
 *   vrfs_ietf_verify_prepared_io_wire_batch: item i is vrfs_ietf_verify_prepared_wire_batch with data[i] = the data of input
 *     input_index[i] as given to vrfs_inputs_prepare - and so vrfs_ietf_verify_wire_batch on the gathered key encodings and data -
 *     ok, hash and status byte for byte, without hash-to-curve per item.  An input index out of range, or an input with
 *     input_ok = 0, is VRFS_ITEM_INVALID_DATA with ok 0 and a zero hash.  The keys must come from vrfs_public_keys_prepare_encoded.
 * Input points come from hash-to-curve and lie in the prime-order subgroup, where the table's s*I equals the s*I of the other
 * calls; O goes through the same variable-base path as there, so this adds no caveat to those above.  Handles follow the rules
 * of prepared keys: one context; orphaned by vrfs_ctx_destroy; release of an orphan or NULL only frees the record.  A keys and an
 * inputs handle of different suites or contexts are VRFS_BAD_ARG.  n = 0 returns VRFS_OK. */
typedef struct vrfs_inputs vrfs_inputs;
vrfs_status vrfs_inputs_prepare(vrfs_ctx*, vrfs_suite, size_t n_inputs, const uint8_t* data, const uint64_t* data_off /*n_inputs+1*/,
                                uint8_t* out_input_ok /*n_inputs, may be NULL*/, uint8_t* out_points /*n_inputs*64, may be NULL*/,
                                vrfs_inputs** out);
void vrfs_inputs_release(vrfs_inputs*);
vrfs_status vrfs_ietf_verify_prepared_io_batch(vrfs_ctx*, const vrfs_public_keys*, const vrfs_inputs*, size_t n, const uint32_t* key_index,
                                               const uint32_t* input_index, const uint8_t* output, const uint8_t* c, const uint8_t* s,
                                               const uint8_t* ad, const uint64_t* ad_off, uint8_t* out_ok, uint8_t* out_status /* may be NULL */);
vrfs_status vrfs_ietf_verify_prepared_io_batch_dev(vrfs_ctx*, const vrfs_public_keys*, const vrfs_inputs*, size_t n, const uint32_t* d_key_index,
                                                   const uint32_t* d_input_index, const uint8_t* d_output, const uint8_t* d_c, const uint8_t* d_s,
                                                   const uint8_t* d_ad, const uint64_t* d_ad_off, uint8_t* d_out_ok, uint8_t* d_out_status /* may be NULL */);
vrfs_status vrfs_ietf_verify_prepared_io_wire_batch(vrfs_ctx*, const vrfs_public_keys*, const vrfs_inputs*, size_t n, const uint32_t* key_index,
                                                    const uint32_t* input_index, const uint8_t* sig /*n*sig_len*/, const uint8_t* ad,
                                                    const uint64_t* ad_off, uint8_t* out_ok, uint8_t* out_hash /*n*hash_len, may be NULL*/,
                                                    uint8_t* out_status /* may be NULL */);

/* pedersen::Prover::prove / Verifier::verify (A.10).  proof = pk_com || r || ok (3 x 64-byte affine) || s || sb (2 x 32 bytes) = 256 bytes. */
vrfs_status vrfs_pedersen_prove_batch(vrfs_ctx*, vrfs_suite, size_t n, const uint8_t* sk, const uint8_t* input, const uint8_t* output,
                                      const uint8_t* ad, const uint64_t* ad_off, uint8_t* out_proof /*n*256*/, uint8_t* out_blinding /*n*32*/);
vrfs_status vrfs_pedersen_verify_batch(vrfs_ctx*, vrfs_suite, size_t n, const uint8_t* input, const uint8_t* output, const uint8_t* proof,
                                       const uint8_t* ad, const uint64_t* ad_off, uint8_t* out_ok, uint8_t* out_status /* may be NULL */);
/* The same with the typed `pedersen::Proof` in its serialised form (its CanonicalSerialize, A.10): point_encode(pk_com) ||
 * point_encode(r) || point_encode(ok) || s || sb in codec byte order - 3 * enc_len + 64 bytes (Bandersnatch: 160 B, the size
 * SURVEY 8b specifies).  verify deserialises like the reference (canonical, on curve, prime-order subgroup, s and sb < r). */
int vrfs_suite_pedersen_proof_len(vrfs_suite s);
vrfs_status vrfs_pedersen_prove_compressed_batch(vrfs_ctx*, vrfs_suite, size_t n, const uint8_t* sk, const uint8_t* input, const uint8_t* output,
                                                 const uint8_t* ad, const uint64_t* ad_off, uint8_t* out_proof /*n*proof_len*/, uint8_t* out_blinding /*n*32*/);
vrfs_status vrfs_pedersen_verify_compressed_batch(vrfs_ctx*, vrfs_suite, size_t n, const uint8_t* input, const uint8_t* output, const uint8_t* proof /*n*proof_len*/,
                                                  const uint8_t* ad, const uint64_t* ad_off, uint8_t* out_ok, uint8_t* out_status /* may be NULL */);

/* Wire formats (SURVEY.md 8f-1): the serialised forms `CanonicalSerialize/Deserialize` (Compress::Yes, Validate::Yes)
 * give `Public`, `Output` and `ietf::Proof` (names at /root/reference/src/lib.rs:13-17), so that keys and signatures
 * can be verified straight off the wire:
 *   encoded point : Codec::point_encode bytes (32 B arkworks / 33 B SEC1); deserialisation = canonical + on curve +
 *                   prime-order subgroup (the reference: ark-ec `mul_bigint(r).is_zero()`; here a 2-descent for
 *                   Bandersnatch, [L]P for Ed25519, nothing for cofactor-1 secp256r1 - same predicate)
 *   proof         : c (CHALLENGE_LEN bytes, codec byte order, reduced mod r) || s (32 bytes, rejected when >= r)
 *   signature     : point_encode(Output) || proof   (Bandersnatch 96 B, Ed25519 80 B, secp256r1 81 B = RFC 9381 pi_string)
 * secp256r1: the wire form is the CODEC's (SEC1 points, big-endian scalars = RFC 9381 pi_string, pinned by the RFC's examples), not
 * necessarily the crate's derived CanonicalSerialize (possibly arkworks' 33-byte little-endian x || flags with little-endian
 * scalars) - unpinned without the crate; see csrc/wire.cuh. */
int vrfs_suite_ietf_signature_len(vrfs_suite s);
vrfs_status vrfs_point_decode_checked_batch(vrfs_ctx*, vrfs_suite, size_t n, const uint8_t* enc, uint8_t* out_pts /*n*64*/, uint8_t* out_ok);
vrfs_status vrfs_subgroup_check_batch(vrfs_ctx*, vrfs_suite, size_t n, const uint8_t* pts /*n*64*/, uint8_t* out_ok);
/* Input::new(data_i) -> Secret::output -> ietf::Prover::prove -> serialise.  out_ok may be NULL (0 = no input point found). */
vrfs_status vrfs_ietf_sign_wire_batch(vrfs_ctx*, vrfs_suite, size_t n, const uint8_t* sk, const uint8_t* data, const uint64_t* data_off,
                                      const uint8_t* ad, const uint64_t* ad_off, uint8_t* out_sig /*n*sig_len*/, uint8_t* out_ok);
/* Public::deserialize + Input::new(data_i) + Output/Proof::deserialize + ietf::Verifier::verify.  out_hash (may be NULL):
 * Output::hash of the accepted items (zero for rejected ones), n*hash_len. */
vrfs_status vrfs_ietf_verify_wire_batch(vrfs_ctx*, vrfs_suite, size_t n, const uint8_t* pk_enc /*n*enc_len*/, const uint8_t* data,
                                        const uint64_t* data_off, const uint8_t* sig /*n*sig_len*/, const uint8_t* ad,
                                        const uint64_t* ad_off, uint8_t* out_ok, uint8_t* out_hash, uint8_t* out_status /* may be NULL */);

/* Pedersen on the wire: signature = point_encode(Output) || point_encode(pk_com) || point_encode(r) || point_encode(ok) || s || sb
 * (an `Output` followed by `pedersen::Proof`'s CanonicalSerialize; Bandersnatch 192 B).  Deserialisation validates all four points
 * (canonical, on curve, prime-order subgroup) and both scalars (canonical).  The blinding factor is returned to the prover only. */
int vrfs_suite_pedersen_signature_len(vrfs_suite s);
vrfs_status vrfs_pedersen_sign_wire_batch(vrfs_ctx*, vrfs_suite, size_t n, const uint8_t* sk, const uint8_t* data, const uint64_t* data_off,
                                          const uint8_t* ad, const uint64_t* ad_off, uint8_t* out_sig /*n*sig_len*/, uint8_t* out_blinding /*n*32*/, uint8_t* out_ok);
vrfs_status vrfs_pedersen_verify_wire_batch(vrfs_ctx*, vrfs_suite, size_t n, const uint8_t* data, const uint64_t* data_off, const uint8_t* sig /*n*sig_len*/,
                                            const uint8_t* ad, const uint64_t* ad_off, uint8_t* out_ok, uint8_t* out_status /* may be NULL */);

/* Batch verification of pedersen::Verifier::verify by one random linear combination (Bandersnatch only).
 * With E_i = Ok_i + c_i O_i - s_i I_i and F_i = R_i + c_i Yb_i - s_i G - sb_i B (both 0 for a valid proof), the batch is accepted
 * iff sum_i rho_i E_i + sigma_i F_i = 0, one multi-scalar multiplication over the 5n + 2 points instead of 2n per-item ones.
 * Coefficients: (rho_i || sigma_i) = the first 32 bytes of SHA-512("vrfs-b200/pedersen-batch/v1" || seed || LE64(i) || c_i), c_i the
 * proof's challenge as 32 little-endian bytes; each 16-byte half is read little-endian with its top bit cleared (rho_i, sigma_i < 2^127).
 * seed: 32 secret bytes, fresh per call (whoever made the proofs must not know them).
 * Every point (I, O, Yb, R, Ok) must lie in the prime-order subgroup, or a torsion component can vanish from the sum; the call tests
 * that for every item and counts a point outside the subgroup as a failure.  Other suites return VRFS_UNSUPPORTED: their cofactor-8
 * subgroup test costs more than the batch saves, and short-Weierstrass curves have no bucket path here.
 * *out_all_ok = 1  => every item verifies (false accept <= 2^-127 per call when the seed is secret);
 * *out_all_ok = 0  => at least one item fails, is invalid, or has a point outside the prime-order subgroup.
 * out_ok / out_status (each may be NULL): all 1 / VRFS_ITEM_OK when *out_all_ok = 1; otherwise the call runs the
 * per-item verifier and returns exactly what vrfs_pedersen_verify_batch returns for the same arguments.
 * n = 0: VRFS_OK with *out_all_ok = 1.  At most 2^24 proofs per call. */
vrfs_status vrfs_pedersen_batch_verify(vrfs_ctx*, vrfs_suite, size_t n, const uint8_t* input, const uint8_t* output,
                                       const uint8_t* proof /*n*256*/, const uint8_t* ad, const uint64_t* ad_off,
                                       const uint8_t* seed /*32*/, uint8_t* out_all_ok, uint8_t* out_ok, uint8_t* out_status);
/* the same from serialised signatures (Output || pedersen::Proof, the layout of vrfs_pedersen_verify_wire_batch); their points are
 * subgroup-checked by the decoder, and out_ok / out_status of a rejected batch are what vrfs_pedersen_verify_wire_batch returns */
vrfs_status vrfs_pedersen_batch_verify_wire(vrfs_ctx*, vrfs_suite, size_t n, const uint8_t* data, const uint64_t* data_off,
                                            const uint8_t* sig /*n*sig_len*/, const uint8_t* ad, const uint64_t* ad_off,
                                            const uint8_t* seed /*32*/, uint8_t* out_all_ok, uint8_t* out_ok, uint8_t* out_status);

/* ring commitment MSM (ark-ec VariableBaseMSM::msm behind ring-proof's KZG commit, SURVEY 3.5):
 * n_columns scalar columns (column-major, n*32 bytes each) over one base vector of n affine G1 points.
 * out: n_columns * 96 bytes affine.
 * Precondition (what a `G1Affine` obtained by validated deserialisation guarantees): the bases lie in the prime-order subgroup G1.
 * The stateless form splits every scalar with G1's endomorphism (k = k1 + q z^2 over [P | -phi(P)]), which equals the plain sum
 * only there; vrfs_g1_decompress_batch(check_subgroup = 1) is the validating loader.  The prepared forms below use no endomorphism. */
vrfs_status vrfs_msm_g1_bls12_381(vrfs_ctx*, size_t n, const uint8_t* bases /*n*96*/, const uint8_t* scalars /*n_columns*n*32*/,
                                  int n_columns, uint8_t* out /*n_columns*96*/);
/* the same with a tuning hint: window_bits (0 = automatic, else 7..16).  The result never depends on it. */
vrfs_status vrfs_msm_g1_bls12_381_ex(vrfs_ctx*, size_t n, const uint8_t* bases /*n*96*/, const uint8_t* scalars /*n_columns*n*32*/, int n_columns, int window_bits,
                                     uint8_t* out /*n_columns*96*/);
/* Prepared bases: the counterpart of `RingContext` holding the SRS.  `prepare` stores 2^(c*w) * P_i for every window
 * once (device memory: ceil(256/c) * n * 96 bytes, affine); `prepared` then computes n_columns commitments with one shared
 * bucket set per column and no Horner chain.  Results are identical to vrfs_msm_g1_bls12_381. */
/* Short SRS (n <= 16384, i.e. ring sizes up to 2^13) prepared WITHOUT hints also get the table of the 128 multiples of every
 * 2^(8w) P_i (393 KB of device memory per base: 0.8 GB at n = 2^11, 6.4 GB at 2^14); a commitment is then the plain sum of the
 * table entries the scalars' signed radix-256 digits select - no sort, no buckets (2^11 x 3 columns: 0.25 ms instead of 0.36).
 * If that allocation fails the handle silently keeps the bucket pipeline.  A window_bits / threads_per_bucket hint
 * (vrfs_msm_g1_prepare_ex) selects the bucket pipeline explicitly. */
typedef struct vrfs_msm_bases vrfs_msm_bases;
vrfs_status vrfs_msm_g1_prepare(vrfs_ctx*, size_t n, const uint8_t* bases /*n*96*/, vrfs_msm_bases** out);
/* the same with tuning hints: window_bits (0 = automatic, else 8..18) and threads_per_bucket (0 = automatic, else a power of two
 * <= 32).  The results never depend on them.  On failure *out stays NULL and nothing is leaked. */
vrfs_status vrfs_msm_g1_prepare_ex(vrfs_ctx*, size_t n, const uint8_t* bases /*n*96*/, int window_bits, int threads_per_bucket, vrfs_msm_bases** out);
vrfs_status vrfs_msm_g1_prepared(vrfs_ctx*, const vrfs_msm_bases* bases, const uint8_t* scalars /*n_columns*n*32*/, int n_columns, uint8_t* out /*n_columns*96*/);
/* the same over this rank's point range, projective partial out (144 B per column) - the multi-GPU form: prepare each rank's
 * slice of the SRS once, all-gather the partials, fold them with vrfs_g1_sum_partials */
vrfs_status vrfs_msm_g1_prepared_partial(vrfs_ctx*, const vrfs_msm_bases* bases, const uint8_t* scalars, int n_columns, uint8_t* out_partial /*n_columns*144*/);
/* May be called before or after vrfs_ctx_destroy of the owning context (destroy frees the tables of handles still alive;
 * releasing such a handle afterwards only frees its record). */
void vrfs_msm_g1_release(vrfs_msm_bases* bases);
/* multi-GPU MSM helper: this rank's partial sums over its point range, projective (X,Y,Z 48-byte LE
 * canonical each = 144 bytes per column), to be gathered (NCCL all-gather of 144*n_columns bytes) and
 * folded with vrfs_g1_sum_partials on any rank. */
vrfs_status vrfs_msm_g1_partial(vrfs_ctx*, size_t n, const uint8_t* bases, const uint8_t* scalars, int n_columns, uint8_t* out_partial /*n_columns*144*/);
vrfs_status vrfs_g1_sum_partials(vrfs_ctx*, int n_parts, int n_columns, const uint8_t* partials /*n_parts*n_columns*144*/, uint8_t* out /*n_columns*96*/);

/* ---- several GPUs of one node (SURVEY.md 8e) -----------------------------------------------------------------------------
 * VRF batches are independent items: they shard by index range and never communicate.  The commitment MSM splits by point
 * range; each GPU reduces its range to one projective partial per column (144 B) and the partials are exchanged by the MSM's
 * last kernel itself: it stores them into the peers' device memory over NVLink (peer access / CUDA IPC), raises a flag behind a
 * system-scope fence, waits for the other ranks' flags in its own memory, adds and normalises.  No NCCL call, no host hop.
 *
 * (1) one process per GPU (torch.distributed / torchrun; the shape bench.py runs in): every rank creates an ordinary context,
 *     calls vrfs_ctx_peer_export, all-gathers the 64-byte handles over its own control plane (host side, once), calls
 *     vrfs_ctx_peer_connect.  The *_allgather entry points are COLLECTIVE: every rank of the group must call them in the same
 *     order; every rank receives the full result.  A rank that waits longer than the timeout (default 2 s) for a peer fails with
 *     VRFS_CUDA_ERROR instead of hanging. */
#define VRFS_PEER_HANDLE_BYTES 64
vrfs_status vrfs_ctx_peer_export(vrfs_ctx*, int rank, int world /* <= 16 */, uint8_t* out_handle /*64*/);
vrfs_status vrfs_ctx_peer_connect(vrfs_ctx*, const uint8_t* handles /*world*64, rank order*/);
vrfs_status vrfs_ctx_peer_set_timeout_ms(vrfs_ctx*, unsigned int ms);
int vrfs_ctx_peer_world(const vrfs_ctx*);   /* 0 = not connected */
/* this rank's scalars (n_columns x its n bases, column-major) over its prepared slice of the SRS -> the full commitments */
vrfs_status vrfs_msm_g1_prepared_allgather(vrfs_ctx*, const vrfs_msm_bases* bases, const uint8_t* scalars, int n_columns, uint8_t* out /*n_columns*96*/);
/* the ring commitment with the domain's rows split over the ranks: arguments as vrfs_ring_commit_rows_partial, full result out */
vrfs_status vrfs_ring_commit_rows_allgather(vrfs_ctx*, const vrfs_msm_bases* srs_rows, size_t row_lo, size_t keyset_part_size, size_t n_keys,
                                            const uint8_t* keys_rows, const uint8_t* padding, size_t n_tail, const uint8_t* tail,
                                            uint8_t* out_commitment /*3*96*/);
/* (2) one caller, several GPUs - the `vrfs_ctx_create(const int* devices, int n_devices, ..)` of SURVEY.md 8b.  The multi-device
 *     context owns one context per device (vrfs_mctx_device_ctx gives them for the per-device entry points), enables peer access
 *     between them, shards verify batches by index range and runs the MSM exchange with device 0 as the folding rank.  Host
 *     buffers should be pinned, otherwise the per-device copies serialise in the driver. */
typedef struct vrfs_mctx vrfs_mctx;
typedef struct vrfs_multi_bases vrfs_multi_bases;
vrfs_status vrfs_ctx_create_multi(const int* devices, int n_devices, vrfs_mctx** out);   /* *out is set even on failure: read the error, then destroy */
void vrfs_mctx_destroy(vrfs_mctx*);
int vrfs_mctx_device_count(const vrfs_mctx*);
vrfs_ctx* vrfs_mctx_device_ctx(vrfs_mctx*, int i);
const char* vrfs_mctx_last_error(const vrfs_mctx*);
uint64_t vrfs_mctx_launch_count(const vrfs_mctx*);
vrfs_status vrfs_multi_ietf_verify_batch(vrfs_mctx*, vrfs_suite, size_t n, const uint8_t* pk, const uint8_t* input, const uint8_t* output,
                                         const uint8_t* c, const uint8_t* s, const uint8_t* ad, const uint64_t* ad_off, uint8_t* out_ok,
                                         uint8_t* out_status /* may be NULL */);
vrfs_status vrfs_multi_msm_g1_prepare(vrfs_mctx*, size_t n, const uint8_t* bases /*n*96*/, vrfs_multi_bases** out);
vrfs_status vrfs_multi_msm_g1_prepared(vrfs_mctx*, const vrfs_multi_bases*, const uint8_t* scalars /*n_columns*n*32*/, int n_columns, uint8_t* out /*n_columns*96*/);
vrfs_status vrfs_multi_ring_commit(vrfs_mctx*, const vrfs_multi_bases* srs_lagrange, size_t keyset_part_size, size_t n_keys, const uint8_t* keys,
                                   const uint8_t* padding, size_t n_tail, const uint8_t* tail, uint8_t* out_commitment /*3*96*/);
void vrfs_multi_msm_g1_release(vrfs_multi_bases*);

/* ---- ring fixed columns and their commitments (SURVEY.md 8f-2) -----------------------------------------------------------
 * What `ring` -> RingContext::verifier_key / prover_key -> ring-proof `index` -> PiopParams::fixed_columns + FixedColumns::commit
 * compute (named at /root/reference/src/lib.rs:13-17; the ring-proof crate itself is not available offline, so the row layout
 * is given by the caller instead of being hard-coded):
 *   row i of the domain (size N, a power of two):  keys[i]                      for i <  n_keys
 *                                                  padding                      for n_keys <= i < keyset_part_size
 *                                                  tail[i - keyset_part_size]   for the next n_tail rows (the powers 2^j * H)
 *                                                  (0, 0)                       after that
 *   columns: xs | ys | selector (1 on the first keyset_part_size rows), N canonical 32-byte LE values of BLS12-381 Fr each.
 * Points are affine x || y (64 B) of the suite whose base field is BLS12-381 Fr (Bandersnatch). */
vrfs_status vrfs_ring_fixed_columns(vrfs_ctx*, size_t domain_size, size_t keyset_part_size, size_t n_keys, const uint8_t* keys /*n_keys*64*/,
                                    const uint8_t* padding /*64*/, size_t n_tail, const uint8_t* tail /*n_tail*64*/,
                                    uint8_t* out_columns /*3*domain_size*32*/);
/* The three KZG commitments (cx, cy, selector) of those columns over a prepared SRS of exactly domain_size G1 points
 * (vrfs_msm_g1_prepare).  srs_is_lagrange != 0: the bases are [L_i(tau)]G1 over the domain (ring-proof's `Ring`, the updatable
 * form) and the columns are committed as they are; 0: the bases are the monomial powers [tau^i]G1 (`index` / `FixedColumns::commit`)
 * and the columns are interpolated first (inverse FFT below).  Both give the same three points.  out: 3 * 96 bytes affine. */
vrfs_status vrfs_ring_commit(vrfs_ctx*, const vrfs_msm_bases* srs, int srs_is_lagrange, size_t keyset_part_size, size_t n_keys,
                             const uint8_t* keys, const uint8_t* padding, size_t n_tail, const uint8_t* tail, uint8_t* out_commitment /*3*96*/);
/* The homomorphic form of the same commitment over a LAGRANGE-basis SRS (what ring-proof's updatable `Ring` does on append):
 * out = [ sum_{i < n_keys} (x_i - pad_x) L_i ,  sum_{i < n_keys} (y_i - pad_y) L_i ]   (2 * 96 bytes affine), so that
 * commit(ring) = commit(ring of padding only) + (delta_x, delta_y, identity): the MSM touches n_keys rows instead of the whole
 * domain (a half-full ring: 2.2 instead of 3.9 ms at 2^17).  The caller adds the points (vrfs_g1_sum_partials with Z = 1). */
vrfs_status vrfs_ring_commit_delta(vrfs_ctx*, const vrfs_msm_bases* srs_lagrange, size_t n_keys, const uint8_t* keys /*n_keys*64*/,
                                   const uint8_t* padding /*64*/, uint8_t* out_delta /*2*96*/);
/* One rank's share of a multi-GPU ring commitment over a Lagrange-basis SRS: srs_rows holds the prepared bases of the rows
 * [row_lo, row_lo + rows) of the domain, keys_rows the keys that fall into those rows (rows row_lo .. min(n_keys, row_lo + rows) - 1;
 * n_keys is the ring size, as in vrfs_ring_commit).  The three projective partial sums (3 * 144 bytes) of all ranks are gathered
 * and folded with vrfs_g1_sum_partials. */
vrfs_status vrfs_ring_commit_rows_partial(vrfs_ctx*, const vrfs_msm_bases* srs_rows, size_t row_lo, size_t keyset_part_size, size_t n_keys,
                                          const uint8_t* keys_rows, const uint8_t* padding, size_t n_tail, const uint8_t* tail,
                                          uint8_t* out_partial /*3*144*/);
/* ark-poly Radix2EvaluationDomain::fft (inverse = 0: coefficients -> evaluations) / ::ifft (inverse != 0) over BLS12-381 Fr for
 * n_columns vectors of 2^log_n canonical 32-byte LE values (values >= r are reduced); group_gen = TWO_ADIC_ROOT_OF_UNITY^(2^(32-log_n)).
 * in and out may be the same buffer. */
vrfs_status vrfs_fr_fft_batch(vrfs_ctx*, int log_n, int n_columns, int inverse, const uint8_t* in /*n_columns*2^log_n*32*/, uint8_t* out);

/* BLS12-381 G1 on the wire (the points of a `RingCommitment`, an SRS file): ark-bls12-381's compressed CanonicalSerialize /
 * validated CanonicalDeserialize, i.e. the zcash encoding - 48 bytes, big-endian x; bit 7 of byte 0 = compressed, bit 6 = infinity,
 * bit 5 = y is the lexicographically larger root.  Points are 96-byte affine LE (zeros = identity) on the other side.
 * decompress: out_ok[i] = 0 (and a zero point) for a missing compression flag, a non-canonical x, an x that is no abscissa, stray bits on
 * an infinity encoding, or - when check_subgroup != 0 - a point outside the prime-order subgroup (endomorphism test). */
vrfs_status vrfs_g1_compress_batch(vrfs_ctx*, size_t n, const uint8_t* points /*n*96*/, uint8_t* out /*n*48*/);
vrfs_status vrfs_g1_decompress_batch(vrfs_ctx*, size_t n, const uint8_t* enc /*n*48*/, int check_subgroup, uint8_t* out_points /*n*96*/, uint8_t* out_ok /*n*/);

/* ---- BLS12-381 pairing and the batched KZG opening check (SURVEY.md 8f-3) -------------------------------------------------
 * What `ring` -> ring-proof's verifier reduces to after its PIOP identities (ark-ec `Bls12::multi_miller_loop` +
 * `final_exponentiation`, reached through the re-exports at /root/reference/src/lib.rs:13-17).  The ring-proof crate is not
 * available offline, so its transcript is NOT restated: the aggregation coefficients r_i are inputs, like the ring's row layout.
 * G2 points: affine x.c0 || x.c1 || y.c0 || y.c1, 48 bytes little-endian each (192 B; zeros = identity).  GT values: the 12 F_q
 * coefficients of the tower F_q12 -> F_q6 -> F_q2 in order (c0.c0.c0, c0.c0.c1, c0.c1.c0, ...), 48 bytes LE each (576 B); the
 * engine's final exponent is 3 (q^12 - 1)/r (the usual x-chain), i.e. its GT values are cubes of the textbook ones.
 *
 * n independent products  prod_{j < n_pairs} e(+-P_ij, Q_ij)  (n_pairs <= 4; bit j of negate_masks[i] negates P_ij; NULL = none):
 * out_ok[i] = 1 if the product is one, 0 if not, 2 if a point is non-canonical or off its curve; out_gt (may be NULL) gets the
 * product's value.  Points are NOT subgroup-checked here. */
vrfs_status vrfs_pairing_product_batch(vrfs_ctx*, size_t n, int n_pairs, const uint8_t* g1 /*n*n_pairs*96*/, const uint8_t* g2 /*n*n_pairs*192*/,
                                       const uint32_t* negate_masks /*n*/, uint8_t* out_ok /*n*/, uint8_t* out_gt /*n*576*/);
/* (check_points 0 and 1 presume that C_i, W_i are in G1, as typed `G1Affine` values are; only level 2 detects a point of the curve outside it.)
 * k KZG openings (commitment C_i, point z_i, value v_i, proof W_i; scalars 32-byte LE, reduced mod r) checked at once against the
 * verifier key (G2, [tau]G2) with aggregation coefficients r_i:  e(sum r_i (C_i - [v_i]G1 + [z_i]W_i), G2) = e(sum r_i W_i, [tau]G2).
 * One 2-column MSM over 2k+1 points + one product of two pairings.  check_points: 0 = C_i, W_i are typed values (already
 * validated), 1 = canonical + on the curve, 2 = also in the prime-order subgroup (what CanonicalDeserialize validates).
 * *out_ok = 1 accepted, 0 rejected, 2 malformed point. */
vrfs_status vrfs_kzg_batch_verify(vrfs_ctx*, size_t k, const uint8_t* commitments /*k*96*/, const uint8_t* points_z /*k*32*/, const uint8_t* values_v /*k*32*/,
                                  const uint8_t* proofs /*k*96*/, const uint8_t* coeffs_r /*k*32*/, const uint8_t* g2 /*192*/, const uint8_t* tau_g2 /*192*/,
                                  int check_points, uint8_t* out_ok /*1*/);

/* self-test / measurement helper: 1/a in BLS12-381 Fq (the inversion behind the MSM's affine output) for n canonical 48-byte LE
 * values, 0 -> 0; out_ok[i] = 1 when the word-approximation GCD finished without falling back to the binary Euclid. */
vrfs_status vrfs_fq381_inv_batch(vrfs_ctx*, size_t n, const uint8_t* in /*n*48*/, uint8_t* out /*n*48*/, uint8_t* out_ok /*n*/);

/* measurement helper: runs the IMAD.WIDE.U32 issue-rate microbenchmark used as the integer-pipe roofline
 * denominator; returns multiply-accumulates (32x32+64) per second over the whole GPU. */
vrfs_status vrfs_measure_mac32_peak(vrfs_ctx*, int variant, double* out_mac_per_s, double* out_sm_mhz_est);

#ifdef __cplusplus
}
#endif
#endif
