// PreparedPublics of include/vrfs_b200.hpp: proofs of 7 known signers verified by key index give the verdicts of Public::verify on
// the gathered keys, a damaged proof and an index out of range fail on their own item only, and a handle outliving its engine is
// released safely.
#include <algorithm>
#include <cstdio>
#include <memory>
#include <string>

#include "../../include/vrfs_b200.hpp"

using namespace vrfs;

static int failures = 0;
#define CHECK(cond) do { if (!(cond)) { std::printf("FAIL %s:%d: %s\n", __FILE__, __LINE__, #cond); failures++; } } while (0)

int main() {
  const size_t n_keys = 7, n = 50;
  std::unique_ptr<PreparedPublics> outlives;
  {
    Engine eng(0);
    Suite suite = Suite::bandersnatch(eng);
    std::vector<Bytes> seeds, alphas, ad;
    for (size_t k = 0; k < n_keys; k++) { std::string t = "signer-" + std::to_string(k); seeds.push_back(Bytes(t.begin(), t.end())); }
    Secret keys = Secret::from_seed(suite, seeds);
    std::vector<uint32_t> index(n);
    Secret signer{suite, Bytes(32 * n), Bytes(64 * n)};     // item i's secret and public key: those of key index[i]
    for (size_t i = 0; i < n; i++) {
      index[i] = (uint32_t)((i * 5 + 3) % n_keys);
      std::copy_n(keys.scalars.begin() + 32 * index[i], 32, signer.scalars.begin() + 32 * i);
      std::copy_n(keys.public_points.begin() + 64 * index[i], 64, signer.public_points.begin() + 64 * i);
      std::string t = "prepared-" + std::to_string(i);
      alphas.push_back(Bytes(t.begin(), t.end()));
      ad.push_back(Bytes(i % 5, (uint8_t)i));
    }
    auto [input, hok] = Input::new_(suite, alphas);
    Output output = signer.output(input);
    ietf::Proof proof = signer.prove(input, output, ad);

    PreparedPublics prepared(keys.public_());
    CHECK(prepared.size() == n_keys);
    for (size_t k = 0; k < n_keys; k++) CHECK(prepared.key_ok()[k] == 1);
    Errors errs;
    Bytes ok = prepared.verify(index, input, output, ad, proof, &errs);
    for (size_t i = 0; i < n; i++) CHECK(ok[i] == 1 && errs[i] == Error::None);

    proof.c[32 * 20] ^= 1;                                    // a damaged challenge
    index[33] = (uint32_t)((index[33] + 1) % n_keys);         // a valid but wrong key
    index[49] = (uint32_t)n_keys;                             // out of range
    ok = prepared.verify(index, input, output, ad, proof, &errs);
    Public gathered{{suite, signer.public_points}};
    std::copy_n(keys.public_points.begin() + 64 * index[33], 64, gathered.xy.begin() + 64 * 33);
    Errors errs1;
    Bytes ok1 = gathered.verify(input, output, ad, proof, &errs1);
    for (size_t i = 0; i < n - 1; i++) CHECK(ok[i] == ok1[i] && errs[i] == errs1[i]);
    for (size_t i = 0; i < n; i++) CHECK(ok[i] == (i != 20 && i != 33 && i != 49));
    CHECK(errs[20] == Error::VerificationFailure && errs[33] == Error::VerificationFailure && errs[49] == Error::InvalidData);

    outlives.reset(new PreparedPublics(keys.public_()));
  }
  outlives.reset();                                           // its engine is gone: releasing the orphan only frees the record
  if (failures) return 1;
  std::printf("all ok\n");
  return 0;
}
