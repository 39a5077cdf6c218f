// Drives Groth16VerifyBatch of playsnark_b200/host/playsnark.hpp on the README circuit's golden key and proof, from a token
// file written by tests/test_host_cpp_verify_batch.py, and prints the decisions for the test to compare.
#include <cstdio>
#include <fstream>
#include <iostream>
#include <string>

#include "../playsnark_b200/host/playsnark.hpp"

using namespace playsnark;

static std::ifstream in;
template <size_t N> static std::array<uint8_t, N> rd() {
  std::string s; in >> s;
  std::array<uint8_t, N> a{};
  if (s.size() != 2 * N) { fprintf(stderr, "bad token length %zu (want %zu)\n", s.size(), 2 * N); exit(2); }
  for (size_t i = 0; i < N; i++) a[i] = (uint8_t)std::stoi(s.substr(2 * i, 2), nullptr, 16);
  return a;
}

int main(int argc, char** argv) {
  if (argc < 2) return 2;
  in.open(argv[1]);
  Groth16VerifKey vk;
  vk.Alpha = rd<48>(); vk.Beta2 = rd<96>(); vk.Gamma = rd<96>(); vk.Delta2 = rd<96>();
  size_t n_io; in >> n_io;
  vk.IoLP.resize(n_io);
  for (auto& p : vk.IoLP) p = rd<48>();
  Groth16Proof p;
  p.A = rd<48>(); p.B = rd<96>(); p.C = rd<48>();
  G1 c_plus_g = rd<48>();
  Vector io(n_io);
  for (auto& v : io) in >> v;
  try {
    Backend be(0);
    Groth16Proof bad = p;
    bad.C = c_plus_g;
    std::vector<bool> verdicts;
    const bool ok = Groth16VerifyBatch(be, vk, {p, p, bad}, {io, io, io}, &verdicts);
    printf("ok %d\nverdicts", ok ? 1 : 0);
    for (bool v : verdicts) printf(" %d", v ? 1 : 0);
    printf("\nhonest %d\n", Groth16VerifyBatch(be, vk, {p, p}, {io, io}) ? 1 : 0);
    printf("single %d\n", Groth16Verify(be, vk, p, io) ? 1 : 0);
    Vector shortio(io.begin(), io.end() - 1);
    try { Groth16VerifyBatch(be, vk, {p}, {shortio}); printf("short none\n"); } catch (const std::invalid_argument&) { printf("short mismatch\n"); }
  } catch (const std::exception& e) {
    fprintf(stderr, "FAILED: %s\n", e.what());
    return 1;
  }
  return 0;
}
