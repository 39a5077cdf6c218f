// Drives PHGR13VerifyBatch of playsnark_b200/host/playsnark.hpp on the README circuit, from a token file written by
// tests/test_host_cpp_phgr13_verify_batch.py (a device setup and proof), and prints the decisions for the test to compare.
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
  PHGR13VerifKey vk;
  vk.av = rd<96>(); vk.aw = rd<48>(); vk.ay = rd<96>(); vk.gamma = rd<96>(); vk.bgamma = rd<48>(); vk.bgamma2 = rd<96>();
  vk.yts = rd<96>();
  size_t diff; in >> diff;
  vk.vs.resize(diff); vk.ws.resize(diff); vk.ys.resize(diff);
  for (auto& p : vk.vs) p = rd<48>();
  for (auto& p : vk.ws) p = rd<96>();
  for (auto& p : vk.ys) p = rd<48>();
  PHGR13Proof p;
  p.hs = rd<48>(); p.vss = rd<48>(); p.yss = rd<48>(); p.vass = rd<48>(); p.wass = rd<48>(); p.yass = rd<48>(); p.gz = rd<48>();
  p.wss = rd<96>();
  G1 hs_plus_g = rd<48>();
  Vector io(diff);
  for (auto& v : io) in >> v;
  try {
    Backend be(0);
    PHGR13Proof bad = p;
    bad.hs = hs_plus_g;
    std::vector<bool> verdicts;
    const bool ok = PHGR13VerifyBatch(be, vk, {p, p, bad}, {io, io, io}, &verdicts);
    printf("ok %d\nverdicts", ok ? 1 : 0);
    for (bool v : verdicts) printf(" %d", v ? 1 : 0);
    printf("\nhonest %d\n", PHGR13VerifyBatch(be, vk, {p, p}, {io, io}) ? 1 : 0);
    printf("single %d\n", PHGR13Verify(be, vk, p, io) ? 1 : 0);
    Vector shortio(io.begin(), io.end() - 1);
    try { PHGR13VerifyBatch(be, vk, {p}, {shortio}); printf("short none\n"); } catch (const std::invalid_argument&) { printf("short mismatch\n"); }
  } catch (const std::exception& e) {
    fprintf(stderr, "FAILED: %s\n", e.what());
    return 1;
  }
  return 0;
}
