// PreparedInputs and the PreparedPublics overloads that take it (include/vrfs_b200.hpp): seals of 7 signers over 3 round inputs,
// verified by author index and input index, give the verdicts, hashes and errors of Public::verify_signatures on the gathered
// encodings and data, and the typed overload those of PreparedPublics::verify on the gathered input points; a damaged signature,
// a wrong input and an input index out of range fail on their own item only.
#include <algorithm>
#include <cstdio>
#include <string>

#include "../../include/vrfs_b200.hpp"

using namespace vrfs;

static int failures = 0;
#define CHECK(cond) do { if (!(cond)) { std::printf("FAIL %s:%d: %s\n", __FILE__, __LINE__, #cond); failures++; } } while (0)

int main() {
  const size_t n_keys = 7, n_inputs = 3, n = 60;
  Engine eng(0);
  Suite suite = Suite::bandersnatch(eng);
  const size_t hl = suite.hash_len();
  std::vector<Bytes> seeds, rounds, datas, ad;
  for (size_t k = 0; k < n_keys; k++) { std::string t = "io-signer-" + std::to_string(k); seeds.push_back(Bytes(t.begin(), t.end())); }
  for (size_t j = 0; j < n_inputs; j++) { std::string t = "io-round-entropy-" + std::to_string(j); rounds.push_back(Bytes(t.begin(), t.end())); }
  Secret keys = Secret::from_seed(suite, seeds);
  Bytes enc = keys.public_().serialize_compressed();
  std::vector<uint32_t> index(n), input_index(n);
  Bytes sk(32 * n);
  for (size_t i = 0; i < n; i++) {
    index[i] = (uint32_t)((i * 5 + 3) % n_keys);
    input_index[i] = (uint32_t)((i * 7 + 1) % n_inputs);
    std::copy_n(keys.scalars.begin() + 32 * index[i], 32, sk.begin() + 32 * i);
    datas.push_back(rounds[input_index[i]]);
    ad.push_back(Bytes(i % 5, (uint8_t)i));
  }
  Packed d(datas), a(ad);
  const size_t sl = (size_t)vrfs_suite_ietf_signature_len(suite.id);
  Bytes sigs(n * sl), sok(n);
  eng.check(vrfs_ietf_sign_wire_batch(eng.ctx(), suite.id, n, sk.data(), d.ptr(), d.off.data(), a.ptr(), a.off.data(), sigs.data(), sok.data()));
  for (size_t i = 0; i < n; i++) CHECK(sok[i] == 1);

  PreparedPublics prepared = PreparedPublics::from_compressed(suite, enc);
  PreparedInputs inputs(suite, rounds);
  CHECK(inputs.size() == n_inputs);
  for (size_t j = 0; j < n_inputs; j++) CHECK(inputs.input_ok()[j] == 1);
  auto [in_new, in_ok] = Input::new_(suite, rounds);
  CHECK(inputs.input().xy == in_new.xy && in_ok == inputs.input_ok());
  Errors errs;
  auto [ok, beta] = prepared.verify_signatures(index, inputs, input_index, sigs, ad, &errs);
  for (size_t i = 0; i < n; i++) CHECK(ok[i] == 1 && errs[i] == Error::None);

  sigs[sl * 20 + 40] ^= 1;                                  // a damaged challenge
  input_index[33] = (uint32_t)((input_index[33] + 1) % n_inputs);   // a valid but wrong input
  input_index[59] = (uint32_t)n_inputs;                     // out of range
  auto [ok1, beta1] = prepared.verify_signatures(index, inputs, input_index, sigs, ad, &errs);
  const size_t L = suite.point_enc_len();
  Bytes gathered(n * L);
  std::vector<Bytes> gdata(n);
  for (size_t i = 0; i < n; i++) {
    std::copy_n(enc.begin() + L * index[i], L, gathered.begin() + L * i);
    gdata[i] = rounds[std::min<size_t>(input_index[i], n_inputs - 1)];
  }
  Errors errs_w;
  auto [ok_w, beta_w] = Public::verify_signatures(suite, gathered, gdata, sigs, ad, &errs_w);
  for (size_t i = 0; i < n - 1; i++) CHECK(ok1[i] == ok_w[i] && errs[i] == errs_w[i]);
  CHECK(std::equal(beta1.begin(), beta1.begin() + hl * (n - 1), beta_w.begin()));
  for (size_t i = 0; i < n; i++) CHECK(ok1[i] == (i != 20 && i != 33 && i != 59));
  CHECK(errs[20] == Error::VerificationFailure && errs[33] == Error::VerificationFailure && errs[59] == Error::InvalidData);
  CHECK(std::all_of(beta1.begin() + hl * 59, beta1.end(), [](uint8_t b) { return b == 0; }));
  CHECK(std::equal(beta1.begin(), beta1.begin() + hl, beta.begin()));

  // the typed overload against PreparedPublics::verify on the gathered input points
  auto [inp, iok] = Input::new_(suite, gdata);
  Secret signer{suite, sk, Bytes(64 * n)};
  Output out = signer.output(inp);
  ietf::Proof proof = signer.prove(inp, out, ad);
  proof.s[32 * 7] ^= 1;                                     // a damaged s
  Errors errs_t, errs_r;
  Bytes ok_t = prepared.verify(index, inputs, input_index, out, ad, proof, &errs_t);
  Bytes ok_r = prepared.verify(index, inp, out, ad, proof, &errs_r);
  for (size_t i = 0; i < n - 1; i++) CHECK(ok_t[i] == ok_r[i] && errs_t[i] == errs_r[i]);
  for (size_t i = 0; i < n; i++) CHECK(ok_t[i] == (i != 7 && i != 59));
  CHECK(errs_t[7] == Error::VerificationFailure && errs_t[59] == Error::InvalidData);
  if (failures) return 1;
  std::printf("all ok\n");
  return 0;
}
