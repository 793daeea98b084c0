// vrfs_b200.hpp - header-only C++17 mirror of the reference's public API for the hot path, over the C ABI of
// vrfs_b200.h.  The reference is Rust (`ark-ec-vrfs` = `ark-vrf` 0.1.0; the names below are the ones re-exported at
// /root/reference/src/lib.rs:13-17: Suite, Secret, Public, Input, Output, ietf, pedersen, codec) and no Rust toolchain exists
// in the build image, so this is the compiled-language host side: same names, same argument meaning, and the reference's
// error behaviour mapped onto batches:
//     Result<(), Error>   ->  std::vector<uint8_t> ok flags (1 = Ok(())) plus, on request, one vrfs::Error per item
//                             (Error::None / VerificationFailure / InvalidData - the variant the crate would return)
//     Option<Input>       ->  Input + ok flags
// Every type holds a BATCH of n values in the ABI's layout (scalars 32 B LE, points affine x||y 64 B LE); every method is one
// call into libvrfs_b200.so.  Whole-call failures (CUDA errors, bad arguments) throw vrfs::CallError - they are never turned
// into a verdict.  There is no CPU implementation behind these classes.
#pragma once
#include <array>
#include <cstdint>
#include <random>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "vrfs_b200.h"

namespace vrfs {

using Bytes = std::vector<uint8_t>;
// ark_vrf::Error per item (vrfs_item_status of the C ABI); None stands for Ok(())
enum class Error : uint8_t { None = VRFS_ITEM_OK, VerificationFailure = VRFS_ITEM_VERIFICATION_FAILURE, InvalidData = VRFS_ITEM_INVALID_DATA };
using Errors = std::vector<Error>;
static_assert(sizeof(Error) == 1, "Errors is handed to the C ABI as a byte array");
inline uint8_t* status_ptr(Errors* e, size_t n) { if (!e) return nullptr; e->assign(n, Error::None); return reinterpret_cast<uint8_t*>(e->data()); }

struct CallError : std::runtime_error {
  vrfs_status status;
  CallError(vrfs_status st, const std::string& msg) : std::runtime_error(msg), status(st) {}
};

// variable-length items (`ad`, VRF input data, seeds): concatenation + n+1 offsets
struct Packed {
  Bytes data;
  std::vector<uint64_t> off;
  Packed() : off(1, 0) {}
  explicit Packed(const std::vector<Bytes>& items) : off(1, 0) {
    for (const auto& b : items) { data.insert(data.end(), b.begin(), b.end()); off.push_back(data.size()); }
  }
  size_t size() const { return off.size() - 1; }
  const uint8_t* ptr() const { return data.empty() ? reinterpret_cast<const uint8_t*>("") : data.data(); }
};

// one context on one GPU (RAII)
class Engine {
 public:
  explicit Engine(int device = 0) {
    vrfs_status st = vrfs_ctx_create(device, &ctx_);
    if (st != VRFS_OK) {
      std::string msg = ctx_ ? vrfs_last_error(ctx_) : "context allocation failed";
      if (ctx_) vrfs_ctx_destroy(ctx_);
      ctx_ = nullptr;
      throw CallError(st, msg);
    }
  }
  ~Engine() { if (ctx_) vrfs_ctx_destroy(ctx_); }
  Engine(const Engine&) = delete;
  Engine& operator=(const Engine&) = delete;
  vrfs_ctx* ctx() const { return ctx_; }
  void check(vrfs_status st) const { if (st != VRFS_OK) throw CallError(st, vrfs_last_error(ctx_)); }

 private:
  vrfs_ctx* ctx_ = nullptr;
};

// Page-locks an existing buffer (e.g. the storage of a long-lived Bytes) for the guard's lifetime (vrfs_host_register): batch calls
// copy from / into such memory beside their kernels instead of staging it synchronously.  Registration is an optimisation only: if
// the driver refuses (`ok()` false), the calls still work on the pageable buffer.
class HostRegistration {
 public:
  HostRegistration(const void* p, size_t bytes) : p_(const_cast<void*>(p)) { ok_ = p_ && bytes && vrfs_host_register(p_, bytes) == VRFS_OK; }
  explicit HostRegistration(const Bytes& b) : HostRegistration(b.data(), b.size()) {}
  ~HostRegistration() { if (ok_) vrfs_host_unregister(p_); }
  HostRegistration(const HostRegistration&) = delete;
  HostRegistration& operator=(const HostRegistration&) = delete;
  bool ok() const { return ok_; }

 private:
  void* p_;
  bool ok_ = false;
};

// ark_vrf::Suite: one ciphersuite bound to one engine
struct Suite {
  vrfs_suite id;
  Engine* engine;
  static Suite bandersnatch(Engine& e) { return {VRFS_BANDERSNATCH_ELL2, &e}; }
  static Suite ed25519(Engine& e) { return {VRFS_ED25519_TAI, &e}; }
  static Suite secp256r1(Engine& e) { return {VRFS_P256_TAI, &e}; }
  size_t challenge_len() const { return (size_t)vrfs_suite_challenge_len(id); }           // Suite::CHALLENGE_LEN
  size_t hash_len() const { return (size_t)vrfs_suite_hash_len(id); }
  size_t point_enc_len() const { return (size_t)vrfs_suite_point_enc_len(id); }
  size_t ietf_signature_len() const { return (size_t)vrfs_suite_ietf_signature_len(id); }
  size_t pedersen_signature_len() const { return (size_t)vrfs_suite_pedersen_signature_len(id); }
  size_t pedersen_proof_len() const { return (size_t)vrfs_suite_pedersen_proof_len(id); }
};

struct Points { Suite suite; Bytes xy; size_t size() const { return xy.size() / 64; } };   // n affine points

struct Input : Points {
  // Input::new(data) = Suite::data_to_point; ok[i] = 0 stands for None
  static std::pair<Input, Bytes> new_(const Suite& s, const std::vector<Bytes>& datas) {
    Packed d(datas); size_t n = d.size();
    Input in{{s, Bytes(64 * n)}}; Bytes ok(n);
    s.engine->check(vrfs_data_to_point_batch(s.engine->ctx(), s.id, n, d.ptr(), d.off.data(), in.xy.data(), ok.data()));
    return {std::move(in), std::move(ok)};
  }
};

struct Output : Points {
  Bytes hash() const {                                   // Output::hash = Suite::point_to_hash
    Bytes h(suite.hash_len() * size());
    suite.engine->check(vrfs_point_to_hash_batch(suite.engine->ctx(), suite.id, size(), xy.data(), h.data()));
    return h;
  }
  Bytes serialize_compressed() const {
    Bytes e(suite.point_enc_len() * size());
    suite.engine->check(vrfs_point_encode_batch(suite.engine->ctx(), suite.id, size(), xy.data(), e.data()));
    return e;
  }
};

namespace ietf {
struct Proof { Bytes c, s; };                            // n x 32-byte little-endian scalars each
}
namespace pedersen {
struct Proof { Bytes raw; };                             // n x 256: pk_com || r || ok (64 B affine each) || s || sb
struct SerializedProof { Bytes bytes; };                 // n x Suite::pedersen_proof_len(): the proof's CanonicalSerialize (160 B for Bandersnatch)
}

struct Public : Points {
  // ietf::Verifier::verify
  Bytes verify(const Input& input, const Output& output, const std::vector<Bytes>& ad, const ietf::Proof& proof, Errors* errors = nullptr) const {
    Packed a(ad); size_t n = size(); Bytes ok(n);
    suite.engine->check(vrfs_ietf_verify_batch(suite.engine->ctx(), suite.id, n, xy.data(), input.xy.data(), output.xy.data(), proof.c.data(),
                                               proof.s.data(), a.ptr(), a.off.data(), ok.data(), status_ptr(errors, n)));
    return ok;
  }
  Bytes serialize_compressed() const {
    Bytes e(suite.point_enc_len() * size());
    suite.engine->check(vrfs_point_encode_batch(suite.engine->ctx(), suite.id, size(), xy.data(), e.data()));
    return e;
  }
  // CanonicalDeserialize with validation: canonical, on curve, prime-order subgroup
  static std::pair<Public, Bytes> deserialize_compressed(const Suite& s, const Bytes& enc) {
    size_t n = enc.size() / s.point_enc_len();
    Public p{{s, Bytes(64 * n)}}; Bytes ok(n);
    s.engine->check(vrfs_point_decode_checked_batch(s.engine->ctx(), s.id, n, enc.data(), p.xy.data(), ok.data()));
    return {std::move(p), std::move(ok)};
  }
  // serialised keys + VRF input data + serialised signatures (Output || ietf::Proof) -> ok flags and Output::hash
  static std::pair<Bytes, Bytes> verify_signatures(const Suite& s, const Bytes& pk_enc, const std::vector<Bytes>& datas, const Bytes& sigs,
                                                   const std::vector<Bytes>& ad, Errors* errors = nullptr) {
    Packed d(datas), a(ad); size_t n = d.size(); Bytes ok(n), beta(n * s.hash_len());
    s.engine->check(vrfs_ietf_verify_wire_batch(s.engine->ctx(), s.id, n, pk_enc.data(), d.ptr(), d.off.data(), sigs.data(), a.ptr(), a.off.data(),
                                                ok.data(), beta.data(), status_ptr(errors, n)));
    return {std::move(ok), std::move(beta)};
  }
};

// Inputs that many proofs share (a lottery or beacon round): Input::new of each data item once, and one fixed-base table per input
// point on the engine's GPU (vrfs_inputs_prepare); PreparedPublics verifies proofs by key index and input index against them.
// The engine must outlive the calls; destroying it first leaves release safe (RAII).
class PreparedInputs {
 public:
  PreparedInputs(const Suite& s, const std::vector<Bytes>& datas) : suite_(s), input_ok_(datas.size()), points_(64 * datas.size()) {
    Packed d(datas);
    suite_.engine->check(vrfs_inputs_prepare(suite_.engine->ctx(), suite_.id, d.size(), d.ptr(), d.off.data(), input_ok_.data(), points_.data(), &h_));
  }
  ~PreparedInputs() { vrfs_inputs_release(h_); }
  PreparedInputs(const PreparedInputs&) = delete;
  PreparedInputs& operator=(const PreparedInputs&) = delete;
  size_t size() const { return input_ok_.size(); }
  const Bytes& input_ok() const { return input_ok_; }        // Input::new's Option: 0 = no point found
  Input input() const { return Input{{suite_, points_}}; }   // the points, as Input::new gives them
  const vrfs_inputs* handle() const { return h_; }

 private:
  Suite suite_;
  Bytes input_ok_, points_;
  vrfs_inputs* h_ = nullptr;
};

// A Public that is reused ("prepare once, verify many"): one fixed-base table per key on the engine's GPU (vrfs_public_keys_prepare),
// proofs verified by key index.  The engine must outlive the calls; destroying it first leaves release safe (RAII).
class PreparedPublics {
 public:
  explicit PreparedPublics(const Public& keys) : suite_(keys.suite), key_ok_(keys.size()) {
    suite_.engine->check(vrfs_public_keys_prepare(suite_.engine->ctx(), suite_.id, keys.size(), keys.xy.data(), key_ok_.data(), &h_));
  }
  ~PreparedPublics() { vrfs_public_keys_release(h_); }
  PreparedPublics(const PreparedPublics&) = delete;
  PreparedPublics& operator=(const PreparedPublics&) = delete;
  size_t size() const { return key_ok_.size(); }
  const Bytes& key_ok() const { return key_ok_; }            // 1 = a key Public::verify accepts
  // ietf::Verifier::verify with pk[i] = keys[key_index[i]]; an index out of range is Error::InvalidData for that item
  Bytes verify(const std::vector<uint32_t>& key_index, const Input& input, const Output& output, const std::vector<Bytes>& ad, const ietf::Proof& proof,
               Errors* errors = nullptr) const {
    Packed a(ad); size_t n = key_index.size(); Bytes ok(n);
    suite_.engine->check(vrfs_ietf_verify_prepared_batch(suite_.engine->ctx(), h_, n, key_index.data(), input.xy.data(), output.xy.data(), proof.c.data(),
                                                         proof.s.data(), a.ptr(), a.off.data(), ok.data(), status_ptr(errors, n)));
    return ok;
  }
  // keys as serialised (n x point_enc_len bytes), each deserialised and subgroup-checked once (vrfs_public_keys_prepare_encoded):
  // key_ok = 0 where Public::deserialize_compressed rejects the encoding or Public::verify rejects the key
  static PreparedPublics from_compressed(const Suite& s, const Bytes& enc) { return PreparedPublics(s, enc); }
  // Public::verify_signatures with pk_enc[i] = the encoding of key key_index[i] -> (ok, Output::hash); only for from_compressed sets
  std::pair<Bytes, Bytes> verify_signatures(const std::vector<uint32_t>& key_index, const std::vector<Bytes>& datas, const Bytes& sigs,
                                            const std::vector<Bytes>& ad, Errors* errors = nullptr) const {
    Packed d(datas), a(ad); size_t n = key_index.size(); Bytes ok(n), beta(n * suite_.hash_len());
    suite_.engine->check(vrfs_ietf_verify_prepared_wire_batch(suite_.engine->ctx(), h_, n, key_index.data(), d.ptr(), d.off.data(), sigs.data(), a.ptr(),
                                                              a.off.data(), ok.data(), beta.data(), status_ptr(errors, n)));
    return {std::move(ok), std::move(beta)};
  }
  // verify with input[i] = the point of prepared input input_index[i]; an input index out of range is Error::InvalidData
  Bytes verify(const std::vector<uint32_t>& key_index, const PreparedInputs& inputs, const std::vector<uint32_t>& input_index, const Output& output,
               const std::vector<Bytes>& ad, const ietf::Proof& proof, Errors* errors = nullptr) const {
    Packed a(ad); size_t n = key_index.size(); Bytes ok(n);
    suite_.engine->check(vrfs_ietf_verify_prepared_io_batch(suite_.engine->ctx(), h_, inputs.handle(), n, key_index.data(), input_index.data(),
                                                            output.xy.data(), proof.c.data(), proof.s.data(), a.ptr(), a.off.data(), ok.data(),
                                                            status_ptr(errors, n)));
    return ok;
  }
  // verify_signatures with datas[i] = the data of prepared input input_index[i] -> (ok, Output::hash); only for from_compressed sets
  std::pair<Bytes, Bytes> verify_signatures(const std::vector<uint32_t>& key_index, const PreparedInputs& inputs, const std::vector<uint32_t>& input_index,
                                            const Bytes& sigs, const std::vector<Bytes>& ad, Errors* errors = nullptr) const {
    Packed a(ad); size_t n = key_index.size(); Bytes ok(n), beta(n * suite_.hash_len());
    suite_.engine->check(vrfs_ietf_verify_prepared_io_wire_batch(suite_.engine->ctx(), h_, inputs.handle(), n, key_index.data(), input_index.data(),
                                                                 sigs.data(), a.ptr(), a.off.data(), ok.data(), beta.data(), status_ptr(errors, n)));
    return {std::move(ok), std::move(beta)};
  }

 private:
  PreparedPublics(const Suite& s, const Bytes& enc) : suite_(s), key_ok_(enc.size() / s.point_enc_len()) {
    suite_.engine->check(vrfs_public_keys_prepare_encoded(suite_.engine->ctx(), suite_.id, key_ok_.size(), enc.data(), key_ok_.data(), &h_));
  }
  Suite suite_;
  Bytes key_ok_;
  vrfs_public_keys* h_ = nullptr;
};

struct Secret {
  Suite suite;
  Bytes scalars;                                         // n x 32
  Bytes public_points;                                   // n x 64
  size_t size() const { return scalars.size() / 32; }
  static Secret from_seed(const Suite& s, const std::vector<Bytes>& seeds) {
    Packed d(seeds); size_t n = d.size();
    Secret k{s, Bytes(32 * n), Bytes(64 * n)};
    s.engine->check(vrfs_secret_from_seed_batch(s.engine->ctx(), s.id, n, d.ptr(), d.off.data(), k.scalars.data(), k.public_points.data()));
    return k;
  }
  Public public_() const { return Public{{suite, public_points}}; }
  Output output(const Input& input) const {              // Secret::output
    Output o{{suite, Bytes(64 * size())}};
    suite.engine->check(vrfs_output_batch(suite.engine->ctx(), suite.id, size(), scalars.data(), input.xy.data(), o.xy.data()));
    return o;
  }
  ietf::Proof prove(const Input& input, const Output& output, const std::vector<Bytes>& ad) const {      // ietf::Prover::prove
    Packed a(ad); size_t n = size(); ietf::Proof p{Bytes(32 * n), Bytes(32 * n)};
    suite.engine->check(vrfs_ietf_prove_batch(suite.engine->ctx(), suite.id, n, scalars.data(), input.xy.data(), output.xy.data(), a.ptr(),
                                              a.off.data(), p.c.data(), p.s.data()));
    return p;
  }
  // pedersen::Prover::prove -> (Proof, blinding factors)
  std::pair<pedersen::Proof, Bytes> pedersen_prove(const Input& input, const Output& output, const std::vector<Bytes>& ad) const {
    Packed a(ad); size_t n = size(); pedersen::Proof p{Bytes(256 * n)}; Bytes bl(32 * n);
    suite.engine->check(vrfs_pedersen_prove_batch(suite.engine->ctx(), suite.id, n, scalars.data(), input.xy.data(), output.xy.data(), a.ptr(),
                                                  a.off.data(), p.raw.data(), bl.data()));
    return {std::move(p), std::move(bl)};
  }
  // the same with the proof already in its serialised (wire) form
  std::pair<pedersen::SerializedProof, Bytes> pedersen_prove_serialized(const Input& input, const Output& output, const std::vector<Bytes>& ad) const {
    Packed a(ad); size_t n = size(); pedersen::SerializedProof p{Bytes(suite.pedersen_proof_len() * n)}; Bytes bl(32 * n);
    suite.engine->check(vrfs_pedersen_prove_compressed_batch(suite.engine->ctx(), suite.id, n, scalars.data(), input.xy.data(), output.xy.data(), a.ptr(),
                                                             a.off.data(), p.bytes.data(), bl.data()));
    return {std::move(p), std::move(bl)};
  }
  // Input::new(data) -> output -> ietf prove -> serialised signatures point_encode(Output) || c || s
  std::pair<Bytes, Bytes> sign(const std::vector<Bytes>& datas, const std::vector<Bytes>& ad) const {
    Packed d(datas), a(ad); size_t n = size(); Bytes sig(n * suite.ietf_signature_len()), ok(n);
    suite.engine->check(vrfs_ietf_sign_wire_batch(suite.engine->ctx(), suite.id, n, scalars.data(), d.ptr(), d.off.data(), a.ptr(), a.off.data(),
                                                  sig.data(), ok.data()));
    return {std::move(sig), std::move(ok)};
  }
};

namespace pedersen {
// pedersen::Verifier::verify (needs no public key)
inline Bytes verify(const Suite& s, const Input& input, const Output& output, const std::vector<Bytes>& ad, const Proof& proof, Errors* errors = nullptr) {
  Packed a(ad); size_t n = input.size(); Bytes ok(n);
  s.engine->check(vrfs_pedersen_verify_batch(s.engine->ctx(), s.id, n, input.xy.data(), output.xy.data(), proof.raw.data(), a.ptr(), a.off.data(), ok.data(),
                                             status_ptr(errors, n)));
  return ok;
}
// Proof::deserialize_compressed (validated) + verify
inline Bytes verify(const Suite& s, const Input& input, const Output& output, const std::vector<Bytes>& ad, const SerializedProof& proof, Errors* errors = nullptr) {
  Packed a(ad); size_t n = input.size(); Bytes ok(n);
  s.engine->check(vrfs_pedersen_verify_compressed_batch(s.engine->ctx(), s.id, n, input.xy.data(), output.xy.data(), proof.bytes.data(), a.ptr(), a.off.data(),
                                                        ok.data(), status_ptr(errors, n)));
  return ok;
}
// all proofs verified together by one random linear combination (vrfs_pedersen_batch_verify; Bandersnatch only): true iff every
// item verifies.  The 32-byte seed comes from std::random_device and is never shown to the caller (whoever made the proofs must not
// know it).  ok / errors (optional): per-item verdicts, all ok when the batch is accepted, else those of verify() above.
inline bool batch_verify(const Suite& s, const Input& input, const Output& output, const std::vector<Bytes>& ad, const Proof& proof,
                         Bytes* ok = nullptr, Errors* errors = nullptr) {
  Packed a(ad); size_t n = input.size();
  std::random_device rd;
  std::array<uint8_t, 32> seed;
  for (size_t i = 0; i < seed.size(); i += 4) { const uint32_t w = rd(); for (int k = 0; k < 4; k++) seed[i + k] = (uint8_t)(w >> (8 * k)); }
  if (ok) ok->assign(n, 0);
  uint8_t all_ok = 0;
  s.engine->check(vrfs_pedersen_batch_verify(s.engine->ctx(), s.id, n, input.xy.data(), output.xy.data(), proof.raw.data(), a.ptr(),
                                             ad.empty() ? nullptr : a.off.data(), seed.data(), &all_ok, ok ? ok->data() : nullptr, status_ptr(errors, n)));
  seed.fill(0);
  return all_ok != 0;
}
}  // namespace pedersen

// the three KZG commitments behind RingContext::verifier_key: one MSM per scalar column over the SRS bases (BLS12-381 G1)
inline Bytes ring_commitment_msm(Engine& e, const Bytes& bases /*n*96*/, const Bytes& scalar_columns /*ncol*n*32*/, int n_columns) {
  size_t n = bases.size() / 96; Bytes out(96 * (size_t)n_columns);
  e.check(vrfs_msm_g1_bls12_381(e.ctx(), n, bases.data(), scalar_columns.data(), n_columns, out.data()));
  return out;
}


// ark-bls12-381's compressed G1 (de)serialisation (zcash format, 48 bytes) for commitments and SRS points; 96-byte affine LE otherwise
inline Bytes g1_serialize_compressed(Engine& e, const Bytes& points /*n*96*/) {
  size_t n = points.size() / 96; Bytes out(48 * n);
  e.check(vrfs_g1_compress_batch(e.ctx(), n, points.data(), out.data()));
  return out;
}
// -> (points, ok flags): ok[i] = 0 stands for the Err(_) of a validated deserialize_compressed
inline std::pair<Bytes, Bytes> g1_deserialize_compressed(Engine& e, const Bytes& enc /*n*48*/, bool check_subgroup = true) {
  size_t n = enc.size() / 48; Bytes pts(96 * n), ok(n);
  e.check(vrfs_g1_decompress_batch(e.ctx(), n, enc.data(), check_subgroup ? 1 : 0, pts.data(), ok.data()));
  return {pts, ok};
}

// ring::RingContext up to the verifier key's commitment (SURVEY.md 8f-2): holds the prepared SRS of one power-of-two domain
// (Lagrange basis [L_i(tau)]G1 or monomial powers [tau^i]G1, 96-byte affine points) and the row layout of the fixed columns:
// keys | padding up to keyset_part_size | tail (the powers 2^j * H of the blinding base) | zero rows; selector = 1 on the key slots.
// [RECALL, unpinned: the ring-proof crate is not available offline] default keyset_part_size = N - 3 (ZK rows) - |tail| - 1.
class RingContext {
 public:
  RingContext(Engine& e, const Bytes& srs_g1, bool lagrange, const Bytes& padding /*64*/, const Bytes& tail /*n_tail*64*/, size_t keyset_part_size = 0)
      : e_(&e), lagrange_(lagrange), padding_(padding), tail_(tail), n_(srs_g1.size() / 96) {
    part_ = keyset_part_size ? keyset_part_size : n_ - 3 - tail.size() / 64 - 1;
    e.check(vrfs_msm_g1_prepare(e.ctx(), n_, srs_g1.data(), &srs_));
  }
  ~RingContext() { if (srs_) vrfs_msm_g1_release(srs_); }
  RingContext(const RingContext&) = delete;
  RingContext& operator=(const RingContext&) = delete;
  size_t domain_size() const { return n_; }
  size_t max_ring_size() const { return part_; }
  // xs | ys | selector, 3 * N canonical 32-byte LE values
  Bytes fixed_columns(const Bytes& public_keys /*n*64*/) const {
    Bytes out(3 * n_ * 32);
    e_->check(vrfs_ring_fixed_columns(e_->ctx(), n_, part_, public_keys.size() / 64, public_keys.data(), padding_.data(), tail_.size() / 64, tail_.data(), out.data()));
    return out;
  }
  // cx | cy | selector, 3 * 96 bytes affine
  Bytes verifier_key_commitment(const Bytes& public_keys) const {
    Bytes out(3 * 96);
    e_->check(vrfs_ring_commit(e_->ctx(), srs_, lagrange_ ? 1 : 0, part_, public_keys.size() / 64, public_keys.data(), padding_.data(), tail_.size() / 64, tail_.data(), out.data()));
    return out;
  }

  // the serialised RingCommitment: three compressed G1 points (144 bytes)
  Bytes ring_commitment_bytes(const Bytes& public_keys) const { return g1_serialize_compressed(*e_, verifier_key_commitment(public_keys)); }
  // Lagrange-basis SRS only: [sum (x_i - pad_x) L_i, sum (y_i - pad_y) L_i] (2 * 96 bytes) - the part of the commitment that depends on
  // the keys; add it to verifier_key_commitment({}) (the ring of padding only, computed once) with vrfs_g1_sum_partials
  Bytes verifier_key_commitment_delta(const Bytes& public_keys) const {
    Bytes out(2 * 96);
    e_->check(vrfs_ring_commit_delta(e_->ctx(), srs_, public_keys.size() / 64, public_keys.data(), padding_.data(), out.data()));
    return out;
  }

 private:
  Engine* e_;
  bool lagrange_;
  Bytes padding_, tail_;
  size_t n_, part_ = 0;
  vrfs_msm_bases* srs_ = nullptr;
};

}  // namespace vrfs
