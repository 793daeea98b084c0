// pedersen::batch_verify of include/vrfs_b200.hpp: an honest batch is accepted, a batch with one wrong `ad` is rejected and its
// per-item verdicts are those of pedersen::verify, and a suite other than Bandersnatch is refused with VRFS_UNSUPPORTED.
#include <cstdio>
#include <string>

#include "../../include/vrfs_b200.hpp"

using namespace vrfs;

static int failures = 0;
#define CHECK(cond) do { if (!(cond)) { std::printf("FAIL %s:%d: %s\n", __FILE__, __LINE__, #cond); failures++; } } while (0)

int main() {
  Engine eng(0);
  Suite suite = Suite::bandersnatch(eng);
  const size_t n = 40;
  std::vector<Bytes> seeds, alphas, ad;
  for (size_t i = 0; i < n; i++) {
    std::string t = "batch-" + std::to_string(i);
    seeds.push_back(Bytes(t.begin(), t.end()));
    alphas.push_back(Bytes(t.rbegin(), t.rend()));
    ad.push_back(Bytes(i % 7, (uint8_t)i));
  }
  Secret secret = Secret::from_seed(suite, seeds);
  auto [input, hok] = Input::new_(suite, alphas);
  Output output = secret.output(input);
  auto [proof, blinding] = secret.pedersen_prove(input, output, ad);
  Bytes ok; Errors errs;
  CHECK(pedersen::batch_verify(suite, input, output, ad, proof, &ok, &errs));
  for (size_t i = 0; i < n; i++) CHECK(ok[i] == 1 && errs[i] == Error::None);
  CHECK(pedersen::batch_verify(suite, input, output, ad, proof));
  std::vector<Bytes> ad2 = ad;
  ad2[n / 2].push_back(0x55);
  CHECK(!pedersen::batch_verify(suite, input, output, ad2, proof, &ok, &errs));
  Errors errs1;
  Bytes ok1 = pedersen::verify(suite, input, output, ad2, proof, &errs1);
  CHECK(ok == ok1 && errs == errs1);
  CHECK(ok[n / 2] == 0 && errs[n / 2] == Error::VerificationFailure);
  bool refused = false;
  try {
    pedersen::batch_verify(Suite::ed25519(eng), input, output, ad, proof);
  } catch (const CallError& e) {
    refused = e.status == VRFS_UNSUPPORTED;
  }
  CHECK(refused);
  if (failures) return 1;
  std::printf("all ok\n");
  return 0;
}
