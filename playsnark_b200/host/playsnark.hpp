// C++ host-side mirror of the reference's proving interface over the C ABI (header-only).
//
// The reference is compiled Go code; where its toolchain is absent this header is the compiled-
// language host layer: same names, argument meaning and error behaviour as package playsnark
//   Groth16Prove(tr, q, sol)        groth16.go:122     PHGR13Prove(ek, qap, solution)  pinochio.go:207
//   QAP::Quotient(sol)              qap.go:151         BlindEval(p, blindedPoint)      algebra.go:348
//   Groth16Verify(vk, p, io)        groth16.go:214     PHGR13Verify(vk, p, io)         pinochio.go:281
//   Groth16VerifyBatch / PHGR13VerifyBatch: many proofs against one key in one combined pairing check
// Scalars are 32-byte big-endian Elements (kyber Scalar.MarshalBinary), points their compressed
// MarshalBinary bytes.  Go panics become C++ exceptions with the same message.  No arithmetic lives
// here: everything is computed by libplaysnark_b200.so on the GPU.
#pragma once
#include <array>
#include <cstdint>
#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/playsnark_b200.h"

namespace playsnark {

using Element = std::array<uint8_t, 32>;
using G1 = std::array<uint8_t, 48>;
using G2 = std::array<uint8_t, 96>;
using Poly = std::vector<Element>;
using Value = int64_t;
using Vector = std::vector<Value>;

inline const char* kOrderHex = "73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001";

// Value.ToFieldElement (curve.go:17-19): SetInt64 reduces mod r, negatives wrap to r - |v|
inline Element ToFieldElement(Value v) {
  static const uint8_t R[32] = {0x73, 0xed, 0xa7, 0x53, 0x29, 0x9d, 0x7d, 0x48, 0x33, 0x39, 0xd8, 0x08, 0x09, 0xa1, 0xd8, 0x05,
                                0x53, 0xbd, 0xa4, 0x02, 0xff, 0xfe, 0x5b, 0xfe, 0xff, 0xff, 0xff, 0xff, 0x00, 0x00, 0x00, 0x01};
  Element e{};
  uint64_t mag = v < 0 ? (uint64_t)(-(v + 1)) + 1 : (uint64_t)v;
  for (int i = 0; i < 8; i++) e[31 - i] = (uint8_t)(mag >> (8 * i));
  if (v < 0) {  // r - mag
    int borrow = 0;
    for (int i = 31; i >= 0; i--) {
      int d = (int)R[i] - (int)e[i] - borrow;
      borrow = d < 0;
      e[i] = (uint8_t)(d + (borrow ? 256 : 0));
    }
  }
  return e;
}

inline void check(int st) {
  if (st == PS_OK) return;
  if (st == PS_ERR_REMAINDER) throw std::runtime_error("apocalypse");                                   // qap.go:159
  if (st == PS_ERR_LENGTH) throw std::length_error("mismatch of length between poly and blinded eval points");  // algebra.go:351
  throw std::runtime_error(std::string("playsnark_b200: ") + ps_strerror(st));
}

class Backend {
 public:
  explicit Backend(int device = 0) { check(ps_ctx_create(device, &ctx_)); }
  ~Backend() { ps_ctx_destroy(ctx_); }
  Backend(const Backend&) = delete;
  Backend& operator=(const Backend&) = delete;
  ps_ctx* ctx() const { return ctx_; }
 private:
  ps_ctx* ctx_ = nullptr;
};

template <class P>
inline std::vector<uint8_t> flatten(const std::vector<P>& v) {
  std::vector<uint8_t> out(v.size() * sizeof(P) + 1);
  for (size_t i = 0; i < v.size(); i++) std::memcpy(out.data() + i * sizeof(P), v[i].data(), sizeof(P));
  return out;
}

// qap.go:10-27
struct QAP {
  size_t nbVars = 0, nbIO = 0, nbGates = 0;
  std::vector<Poly> left, right, out;
  Poly z;
};

class ResidentQAP {
 public:
  ResidentQAP(Backend& b, const QAP& q) : b_(b), n_(q.nbGates), m_(q.nbVars) {
    auto flat = [&](const std::vector<Poly>& ps) {
      std::vector<uint8_t> o;
      for (auto& p : ps) {
        if (p.size() != q.nbGates) throw std::invalid_argument("QAP polynomial length");
        auto f = flatten(p);
        o.insert(o.end(), f.begin(), f.end() - 1);
      }
      o.push_back(0);
      return o;
    };
    if (q.left.size() != q.nbVars || q.right.size() != q.nbVars || q.out.size() != q.nbVars)
      throw std::invalid_argument("different number of solution variables than polynomials");  // qap.go:177-189
    auto l = flat(q.left), r = flat(q.right), o = flat(q.out), z = flatten(q.z);
    check(ps_qap_load_dense(b.ctx(), q.nbGates, q.nbVars, q.nbIO, l.data(), r.data(), o.data(), z.data(), &h_));
  }
  ~ResidentQAP() { ps_qap_free(h_); }
  // QAP.Quotient, qap.go:151-162
  Poly Quotient(const Vector& sol) const {
    if (sol.size() != m_) throw std::invalid_argument("different number of solution variables than left polynomials");
    Poly w(sol.size());
    for (size_t i = 0; i < sol.size(); i++) w[i] = ToFieldElement(sol[i]);
    auto wb = flatten(w);
    std::vector<uint8_t> hb((n_ - 1) * 32 + 1);
    check(ps_quotient(b_.ctx(), h_, wb.data(), hb.data(), nullptr));
    Poly h(n_ - 1);
    for (size_t i = 0; i + 1 < n_; i++) std::memcpy(h[i].data(), hb.data() + 32 * i, 32);
    return h;
  }
  ps_qap* handle() const { return h_; }
  size_t nbVars() const { return m_; }
 private:
  Backend& b_;
  size_t n_, m_;
  ps_qap* h_ = nullptr;
};

// Poly.BlindEval, algebra.go:348-359, against a resident []Commit
class BlindedPoints {
 public:
  BlindedPoints(Backend& b, const std::vector<G1>& pts) : b_(b) {
    auto f = flatten(pts);
    check(ps_bases_load(b.ctx(), PS_G1, f.data(), pts.size(), PS_FMT_COMPRESSED, 0, 1, &h_));
  }
  ~BlindedPoints() { ps_bases_free(h_); }
  G1 BlindEval(const Poly& p) const {
    auto f = flatten(p);
    G1 out{};
    check(ps_msm(b_.ctx(), h_, f.data(), p.size(), out.data()));
    return out;
  }
 private:
  Backend& b_;
  ps_bases* h_ = nullptr;
};

// groth16.go:30-61 (prover-side fields)
struct Groth16Setup {
  G1 Alpha{}, Beta{}, Delta{};
  std::vector<G1> Xi, NioLP, XiT;
  G2 Beta2{}, Delta2{};
  std::vector<G2> Xi2;
};
struct Groth16Proof {  // groth16.go:106-118
  Element R{}, S{};    // tp
  G1 A{};
  G2 B{};
  G1 C{};
};

class Groth16Prover {
 public:
  Groth16Prover(Backend& b, const Groth16Setup& tr) : b_(b) {
    if (tr.Xi2.size() != tr.Xi.size() || tr.XiT.size() + 1 != tr.Xi.size())
      throw std::length_error("mismatch of length between poly and blinded eval points");
    auto xi = flatten(tr.Xi), xi2 = flatten(tr.Xi2), xit = flatten(tr.XiT), nio = flatten(tr.NioLP);
    check(ps_g16_key_load(b.ctx(), tr.Xi.size(), tr.NioLP.size(), PS_FMT_COMPRESSED, xi.data(), xi2.data(), xit.data(), nio.data(),
                          tr.Alpha.data(), tr.Beta.data(), tr.Delta.data(), tr.Beta2.data(), tr.Delta2.data(), &k_));
  }
  ~Groth16Prover() { ps_g16_key_free(k_); }
  // Groth16Prove, groth16.go:122-211; r, s are the blinding scalars (sampled by the caller as
  // groth16.go:148,158 and kept in the proof's tp)
  Groth16Proof Prove(const ResidentQAP& q, const Vector& sol, const Element& r, const Element& s) const {
    if (sol.size() != q.nbVars()) throw std::invalid_argument("different number of solution variables than left polynomials");
    Poly w(sol.size());
    for (size_t i = 0; i < sol.size(); i++) w[i] = ToFieldElement(sol[i]);
    auto wb = flatten(w);
    Groth16Proof p;
    p.R = r; p.S = s;
    check(ps_g16_prove(b_.ctx(), k_, q.handle(), wb.data(), r.data(), s.data(), p.A.data(), p.B.data(), p.C.data(), nullptr));
    return p;
  }
 private:
  Backend& b_;
  ps_g16_key* k_ = nullptr;
};

// pinochio.go:37-62
struct PHGR13EvalKey {
  std::vector<G1> vs, ys, vas, was, yas, gsi, vbs, wbs, ybs;
  std::vector<G2> ws;
};
struct PHGR13Proof {  // pinochio.go:180-203
  G1 vss{}, vass{}, wass{}, yss{}, yass{}, hs{}, gz{};
  G2 wss{};
};

class PHGR13Prover {
 public:
  PHGR13Prover(Backend& b, const PHGR13EvalKey& ek) : b_(b) {
    auto gsi = flatten(ek.gsi), vs = flatten(ek.vs), ws = flatten(ek.ws), ys = flatten(ek.ys), vas = flatten(ek.vas),
         was = flatten(ek.was), yas = flatten(ek.yas), vbs = flatten(ek.vbs), wbs = flatten(ek.wbs), ybs = flatten(ek.ybs);
    check(ps_phgr13_key_load(b.ctx(), ek.gsi.size() + 1, ek.vs.size(), PS_FMT_COMPRESSED, gsi.data(), vs.data(), ws.data(), ys.data(),
                             vas.data(), was.data(), yas.data(), vbs.data(), wbs.data(), ybs.data(), &k_));
  }
  ~PHGR13Prover() { ps_phgr13_key_free(k_); }
  // PHGR13Prove, pinochio.go:207-254
  PHGR13Proof Prove(const ResidentQAP& q, const Vector& solution) const {
    Poly w(solution.size());
    for (size_t i = 0; i < solution.size(); i++) w[i] = ToFieldElement(solution[i]);
    auto wb = flatten(w);
    uint8_t out[432];
    check(ps_phgr13_prove(b_.ctx(), k_, q.handle(), wb.data(), out, nullptr));
    PHGR13Proof p;
    G1* order[7] = {&p.hs, &p.vss, &p.yss, &p.vass, &p.wass, &p.yass, &p.gz};
    for (int i = 0; i < 7; i++) std::memcpy(order[i]->data(), out + 48 * i, 48);
    std::memcpy(p.wss.data(), out + 336, 96);
    return p;
  }
 private:
  Backend& b_;
  ps_phgr13_key* k_ = nullptr;
};

// ---- verifiers --------------------------------------------------------------------------------------------------
// Groth16Verify, groth16.go:214-233: the verifier side of the setup (IoLP over the public variables, Gamma) and the
// public part of the solution, io[i] for IoLP[i]
struct Groth16VerifKey {
  G1 Alpha{};
  G2 Beta2{}, Gamma{}, Delta2{};
  std::vector<G1> IoLP;
};
inline bool Groth16Verify(Backend& b, const Groth16VerifKey& vk, const Groth16Proof& p, const Vector& io) {
  if (io.size() < vk.IoLP.size()) throw std::invalid_argument("different number of public inputs than IoLP elements");
  Poly w(vk.IoLP.size());
  for (size_t i = 0; i < w.size(); i++) w[i] = ToFieldElement(io[i]);
  auto iolp = flatten(vk.IoLP), wb = flatten(w);
  int ok = 0;
  check(ps_g16_verify(b.ctx(), vk.Alpha.data(), vk.Beta2.data(), vk.Gamma.data(), vk.Delta2.data(), iolp.data(), vk.IoLP.size(), wb.data(),
                      p.A.data(), p.B.data(), p.C.data(), &ok));
  return ok == 1;
}
// Groth16Verify for many proofs against one key as ONE combined pairing-product check with random 128-bit weights drawn
// by the library (ps_g16_verify_batch).  True iff every proof verifies; per_proof (optional) receives one verdict per proof.
inline bool Groth16VerifyBatch(Backend& b, const Groth16VerifKey& vk, const std::vector<Groth16Proof>& proofs,
                               const std::vector<Vector>& ios, std::vector<bool>* per_proof = nullptr) {
  const size_t n = proofs.size(), n_io = vk.IoLP.size();
  if (ios.size() != n) throw std::invalid_argument("different number of proofs than public input vectors");
  Poly w;
  w.reserve(n * n_io);
  std::vector<G1> A, C;
  std::vector<G2> B;
  for (size_t i = 0; i < n; i++) {
    if (ios[i].size() < n_io) throw std::invalid_argument("different number of public inputs than IoLP elements");
    for (size_t j = 0; j < n_io; j++) w.push_back(ToFieldElement(ios[i][j]));
    A.push_back(proofs[i].A); B.push_back(proofs[i].B); C.push_back(proofs[i].C);
  }
  auto iolp = flatten(vk.IoLP), wb = flatten(w), ab = flatten(A), bb = flatten(B), cb = flatten(C);
  std::vector<uint8_t> verdicts(n);
  int ok = 0;
  check(ps_g16_verify_batch(b.ctx(), vk.Alpha.data(), vk.Beta2.data(), vk.Gamma.data(), vk.Delta2.data(), iolp.data(), n_io, n,
                            wb.data(), ab.data(), bb.data(), cb.data(), nullptr, &ok, per_proof ? verdicts.data() : nullptr));
  if (per_proof) per_proof->assign(verdicts.begin(), verdicts.end());
  return ok == 1;
}
// PHGR13Verify, pinochio.go:281-375; vs / ws / ys = the commitments of the public variables (vk.vs[:diff] ...)
struct PHGR13VerifKey {  // pinochio.go:66-90
  G2 av{}, ay{}, gamma{}, bgamma2{}, yts{};
  G1 aw{}, bgamma{};
  std::vector<G1> vs, ys;
  std::vector<G2> ws;
};
inline bool PHGR13Verify(Backend& b, const PHGR13VerifKey& vk, const PHGR13Proof& p, const Vector& io) {
  const size_t diff = vk.vs.size();
  if (vk.ws.size() != diff || vk.ys.size() != diff || io.size() < diff)
    throw std::invalid_argument("different number of public inputs than verification-key elements");
  uint8_t fixed[576], proof[432];
  std::memcpy(fixed, vk.av.data(), 96); std::memcpy(fixed + 96, vk.aw.data(), 48); std::memcpy(fixed + 144, vk.ay.data(), 96);
  std::memcpy(fixed + 240, vk.gamma.data(), 96); std::memcpy(fixed + 336, vk.bgamma.data(), 48);
  std::memcpy(fixed + 384, vk.bgamma2.data(), 96); std::memcpy(fixed + 480, vk.yts.data(), 96);
  const G1* order[7] = {&p.hs, &p.vss, &p.yss, &p.vass, &p.wass, &p.yass, &p.gz};
  for (int i = 0; i < 7; i++) std::memcpy(proof + 48 * i, order[i]->data(), 48);
  std::memcpy(proof + 336, p.wss.data(), 96);
  Poly w(diff);
  for (size_t i = 0; i < diff; i++) w[i] = ToFieldElement(io[i]);
  auto vs = flatten(vk.vs), ws = flatten(vk.ws), ys = flatten(vk.ys), wb = flatten(w);
  int ok = 0;
  check(ps_phgr13_verify(b.ctx(), fixed, vs.data(), ws.data(), ys.data(), diff, wb.data(), proof, &ok));
  return ok == 1;
}
// PHGR13Verify for many proofs against one key in one combined pairing check (ps_phgr13_verify_batch, weights drawn by
// the library); per_proof (optional) receives one verdict per proof
inline bool PHGR13VerifyBatch(Backend& b, const PHGR13VerifKey& vk, const std::vector<PHGR13Proof>& proofs,
                              const std::vector<Vector>& ios, std::vector<bool>* per_proof = nullptr) {
  const size_t n = proofs.size(), diff = vk.vs.size();
  if (vk.ws.size() != diff || vk.ys.size() != diff)
    throw std::invalid_argument("different number of public inputs than verification-key elements");
  if (ios.size() != n) throw std::invalid_argument("different number of proofs than public input vectors");
  uint8_t fixed[576];
  std::memcpy(fixed, vk.av.data(), 96); std::memcpy(fixed + 96, vk.aw.data(), 48); std::memcpy(fixed + 144, vk.ay.data(), 96);
  std::memcpy(fixed + 240, vk.gamma.data(), 96); std::memcpy(fixed + 336, vk.bgamma.data(), 48);
  std::memcpy(fixed + 384, vk.bgamma2.data(), 96); std::memcpy(fixed + 480, vk.yts.data(), 96);
  std::vector<uint8_t> blob(432 * n);
  Poly w;
  w.reserve(n * diff);
  for (size_t i = 0; i < n; i++) {
    if (ios[i].size() < diff) throw std::invalid_argument("different number of public inputs than verification-key elements");
    for (size_t j = 0; j < diff; j++) w.push_back(ToFieldElement(ios[i][j]));
    const PHGR13Proof& p = proofs[i];
    const G1* order[7] = {&p.hs, &p.vss, &p.yss, &p.vass, &p.wass, &p.yass, &p.gz};
    for (int k = 0; k < 7; k++) std::memcpy(blob.data() + 432 * i + 48 * k, order[k]->data(), 48);
    std::memcpy(blob.data() + 432 * i + 336, p.wss.data(), 96);
  }
  auto vs = flatten(vk.vs), ws = flatten(vk.ws), ys = flatten(vk.ys), wb = flatten(w);
  std::vector<uint8_t> verdicts(n);
  int ok = 0;
  check(ps_phgr13_verify_batch(b.ctx(), fixed, vs.data(), ws.data(), ys.data(), diff, n, wb.data(), blob.data(), nullptr, &ok,
                               per_proof ? verdicts.data() : nullptr));
  if (per_proof) per_proof->assign(verdicts.begin(), verdicts.end());
  return ok == 1;
}

}  // namespace playsnark
