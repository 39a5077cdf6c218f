// Wire formats <-> device limbs.
//
// The Go side marshals with kyber's MarshalBinary (used by the reference at pinochio.go:256-275):
// Fr = 32 B big-endian; G1 = 48 B / G2 = 96 B zcash-compressed (bit7 compressed, bit6 infinity,
// bit5 "y is the lexicographically larger root"; Fp2 ordered by c1 then c0 and serialised c1||c0).
// Bulk keys may also come zcash-uncompressed (96 B / 192 B).  All conversion, including the square
// roots of decompression, runs on the device.
#pragma once
#include "group_ops.cuh"

namespace ps {

PS_DEV uint32_t load_be32(const uint8_t* p) {
  return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | (uint32_t)p[3];
}
PS_DEV void store_be32(uint8_t* p, uint32_t v) {
  p[0] = (uint8_t)(v >> 24); p[1] = (uint8_t)(v >> 16); p[2] = (uint8_t)(v >> 8); p[3] = (uint8_t)v;
}

// big-endian bytes (4*N) -> little-endian limbs; `mask_top` clears the three flag bits
template <int N>
PS_DEV void limbs_from_be(uint32_t* v, const uint8_t* b, bool mask_top) {
#pragma unroll
  for (int j = 0; j < N; j++) v[j] = load_be32(b + 4 * (N - 1 - j));
  if (mask_top) v[N - 1] &= 0x1FFFFFFFu;
}
template <int N>
PS_DEV void limbs_to_be(uint8_t* b, const uint32_t* v) {
#pragma unroll
  for (int j = 0; j < N; j++) store_be32(b + 4 * (N - 1 - j), v[j]);
}

// a < MOD ?
template <class P>
PS_DEV bool limbs_lt_mod(const uint32_t* v) {
  uint32_t t = ptx_sub_cc(v[0], P::MOD(0));
#pragma unroll
  for (int j = 1; j < P::N; j++) t = ptx_subc_cc(v[j], P::MOD(j));
  (void)t;
  return ptx_subc(0, 0) != 0;  // borrow <=> v < MOD
}

// standard-form y > (p-1)/2 ?
PS_DEV bool fp_is_larger(const Fp& y_std) {
  uint32_t t = ptx_sub_cc(FpParams::HALF(0), y_std.v[0]);
#pragma unroll
  for (int j = 1; j < 12; j++) t = ptx_subc_cc(FpParams::HALF(j), y_std.v[j]);
  (void)t;
  return ptx_subc(0, 0) != 0;
}
PS_DEV bool fp2_is_larger(const Fp2& y_std) {
  return y_std.c1.is_zero() ? fp_is_larger(y_std.c0) : fp_is_larger(y_std.c1);
}

// ---- Fr ------------------------------------------------------------------------------------------
struct FrFromBytesK {  // 32 B big-endian -> 8 limbs (standard form, or Montgomery when mont != 0)
  static constexpr int BLOCK = 256;
  PS_DEV static void run(uint32_t i, const uint8_t* in, uint32_t* out, int mont, uint32_t* err) {
    Fr x;
    limbs_from_be<8>(x.v, in + (size_t)i * 32, false);
    if (!limbs_lt_mod<FrParams>(x.v)) ps_atomic_or(err, 1u);
    if (mont) x = x.to_mont();
#pragma unroll
    for (int j = 0; j < 8; j++) out[(size_t)i * 8 + j] = x.v[j];
  }
};
struct FrToBytesK {
  static constexpr int BLOCK = 256;
  PS_DEV static void run(uint32_t i, const uint32_t* in, uint8_t* out, int mont) {
    Fr x;
#pragma unroll
    for (int j = 0; j < 8; j++) x.v[j] = in[(size_t)i * 8 + j];
    if (mont) x = x.from_mont();
    limbs_to_be<8>(out + (size_t)i * 32, x.v);
  }
};

// ---- square roots -----------------------------------------------------------------------------------
PS_DEV bool fp_sqrt(const Fp& a, Fp& out) {
  out = fp_sqrt_candidate(a);
  return out.sqr() == a;
}
inline PS_NOINLINE Fp2 fp2_pow(const Fp2& a, const uint32_t* e, int nlimbs) {
  Fp2 acc = Fp2::one();
  bool started = false;
  for (int i = nlimbs - 1; i >= 0; i--) {
    uint32_t w = e[i];
#pragma unroll 1
    for (int b = 31; b >= 0; b--) {
      if (started) acc = acc.sqr();
      if ((w >> b) & 1) { if (started) acc = acc * a; else { acc = a; started = true; } }
    }
  }
  return acc;
}
// complex-method square root in Fp2 (p = 3 mod 4)
PS_DEV bool fp2_sqrt(const Fp2& a, Fp2& out) {
  if (a.is_zero()) { out = a; return true; }
  Fp2 a1 = fp2_pow(a, PS_CEXP(c_FP_P_M3_D4), 12);
  Fp2 alpha = a1.sqr() * a;
  Fp2 x0 = a1 * a;
  Fp2 minus_one = Fp2{Fp::one().neg(), Fp::zero()};
  if (alpha == minus_one) {
    out = Fp2{x0.c1.neg(), x0.c0};  // u * x0
  } else {
    Fp2 b = fp2_pow(alpha + Fp2::one(), PS_CEXP(c_FP_P_M1_D2), 12);
    out = b * x0;
  }
  return out.sqr() == a;
}

PS_DEV Fp fp_curve_rhs(const Fp& x) { return x.sqr() * x + Fp::from_const<FpParams::B_G1>(); }
PS_DEV Fp2 fp_curve_rhs(const Fp2& x) {
  Fp four = Fp::from_const<FpParams::B_G1>();
  return x.sqr() * x + Fp2{four, four};  // b' = 4(1+u)
}

// ---- point decode ------------------------------------------------------------------------------------
PS_DEV bool read_fp(const uint8_t* b, bool mask, Fp& out) {
  Fp t;
  limbs_from_be<12>(t.v, b, mask);
  bool ok = limbs_lt_mod<FpParams>(t.v);
  out = t.to_mont();
  return ok;
}

// r * P == O ?  (kilic's FromCompressed / FromBytes reject points outside the prime-order subgroup; the
// MSM relies on it when it folds k > r/2 to r - k with the point negated)
template <class F>
PS_NOINLINE bool in_subgroup(const Affine<F>& p) {
  uint32_t k[8];
#pragma unroll
  for (int j = 0; j < 8; j++) k[j] = FrParams::MOD(j);
  return xyzz_scalar_mul(XYZZ<F>::from_affine(p), k, 8).is_inf();
}
// the infinity encoding must be canonical: flag bits 0xC0 (compressed) / 0x40 (uncompressed), all else zero
PS_DEV bool inf_is_canonical(const uint8_t* b, int len, bool compressed) {
  uint32_t o = (uint32_t)(b[0] ^ (compressed ? 0xC0 : 0x40));
  for (int k = 1; k < len; k++) o |= b[k];
  return o == 0;
}

// A point that fails is stored as infinity; its error bits (2 = bad encoding / off the curve, 4 = outside the subgroup) are
// OR-ed into *err and, when `status` is given, written to status[i] (0 for a good point).
struct G1DecodeK {
  static constexpr int BLOCK = 128;
  PS_DEV static void run(uint32_t i, const uint8_t* in, int format, G1Affine* out, uint32_t* err, int subgroup, uint8_t* status) {
    const uint8_t* b = in + (size_t)i * (format == PS_FMT_COMPRESSED ? 48 : 96);
    uint8_t flags = b[0];
    bool ok = true;
    G1Affine p = G1Affine::inf();
    if (flags & 0x40) ok = inf_is_canonical(b, format == PS_FMT_COMPRESSED ? 48 : 96, format == PS_FMT_COMPRESSED);
    if (format == PS_FMT_COMPRESSED) {
      if (!(flags & 0x80)) ok = false;
      if (!(flags & 0x40)) {
        Fp x, y;
        ok = read_fp(b, true, x) && ok;
        ok = fp_sqrt(fp_curve_rhs(x), y) && ok;
        bool larger = fp_is_larger(y.from_mont());
        if (larger != ((flags & 0x20) != 0)) y = y.neg();
        p = G1Affine{x, y};
      }
    } else {
      if (flags & 0x80) ok = false;
      if (!(flags & 0x40)) {
        Fp x, y;
        ok = read_fp(b, true, x) && ok;
        ok = read_fp(b + 48, false, y) && ok;
        ok = (y.sqr() == fp_curve_rhs(x)) && ok;
        p = G1Affine{x, y};
      }
    }
    uint32_t e = 0;
    if (!ok) e = 2u;
    else if (subgroup && !p.is_inf() && !in_subgroup(p)) e = 4u;
    if (e) { ps_atomic_or(err, e); p = G1Affine::inf(); }
    if (status) status[i] = (uint8_t)e;
    out[i] = p;
  }
};

struct G2DecodeK {
  static constexpr int BLOCK = 64;
  PS_DEV static void run(uint32_t i, const uint8_t* in, int format, G2Affine* out, uint32_t* err, int subgroup, uint8_t* status) {
    const uint8_t* b = in + (size_t)i * (format == PS_FMT_COMPRESSED ? 96 : 192);
    uint8_t flags = b[0];
    bool ok = true;
    G2Affine p = G2Affine::inf();
    if (flags & 0x40) ok = inf_is_canonical(b, format == PS_FMT_COMPRESSED ? 96 : 192, format == PS_FMT_COMPRESSED);
    if (format == PS_FMT_COMPRESSED) {
      if (!(flags & 0x80)) ok = false;
      if (!(flags & 0x40)) {
        Fp2 x, y;
        ok = read_fp(b, true, x.c1) && ok;
        ok = read_fp(b + 48, false, x.c0) && ok;
        ok = fp2_sqrt(fp_curve_rhs(x), y) && ok;
        Fp2 ys = Fp2{y.c0.from_mont(), y.c1.from_mont()};
        if (fp2_is_larger(ys) != ((flags & 0x20) != 0)) y = y.neg();
        p = G2Affine{x, y};
      }
    } else {
      if (flags & 0x80) ok = false;
      if (!(flags & 0x40)) {
        Fp2 x, y;
        ok = read_fp(b, true, x.c1) && ok;
        ok = read_fp(b + 48, false, x.c0) && ok;
        ok = read_fp(b + 96, false, y.c1) && ok;
        ok = read_fp(b + 144, false, y.c0) && ok;
        ok = (y.sqr() == fp_curve_rhs(x)) && ok;
        p = G2Affine{x, y};
      }
    }
    uint32_t e = 0;
    if (!ok) e = 2u;
    else if (subgroup && !p.is_inf() && !in_subgroup(p)) e = 4u;
    if (e) { ps_atomic_or(err, e); p = G2Affine::inf(); }
    if (status) status[i] = (uint8_t)e;
    out[i] = p;
  }
};

// ---- point encode ------------------------------------------------------------------------------------
PS_DEV void g1_encode(const G1Affine& p, int format, uint8_t* b) {
  int len = format == PS_FMT_COMPRESSED ? 48 : 96;
  if (p.is_inf()) {
    for (int k = 0; k < len; k++) b[k] = 0;
    b[0] = format == PS_FMT_COMPRESSED ? 0xC0 : 0x40;
    return;
  }
  Fp x = p.x.from_mont(), y = p.y.from_mont();
  limbs_to_be<12>(b, x.v);
  if (format == PS_FMT_COMPRESSED) b[0] |= 0x80 | (fp_is_larger(y) ? 0x20 : 0);
  else limbs_to_be<12>(b + 48, y.v);
}
PS_DEV void g2_encode(const G2Affine& p, int format, uint8_t* b) {
  int len = format == PS_FMT_COMPRESSED ? 96 : 192;
  if (p.is_inf()) {
    for (int k = 0; k < len; k++) b[k] = 0;
    b[0] = format == PS_FMT_COMPRESSED ? 0xC0 : 0x40;
    return;
  }
  Fp2 x = Fp2{p.x.c0.from_mont(), p.x.c1.from_mont()};
  Fp2 y = Fp2{p.y.c0.from_mont(), p.y.c1.from_mont()};
  limbs_to_be<12>(b, x.c1.v);
  limbs_to_be<12>(b + 48, x.c0.v);
  if (format == PS_FMT_COMPRESSED) b[0] |= 0x80 | (fp2_is_larger(y) ? 0x20 : 0);
  else { limbs_to_be<12>(b + 96, y.c1.v); limbs_to_be<12>(b + 144, y.c0.v); }
}
PS_DEV void point_encode(const G1Affine& p, int format, uint8_t* b) { g1_encode(p, format, b); }
PS_DEV void point_encode(const G2Affine& p, int format, uint8_t* b) { g2_encode(p, format, b); }
template <class F> struct DecodeKernel;
template <> struct DecodeKernel<Fp> { using K = G1DecodeK; };
template <> struct DecodeKernel<Fp2> { using K = G2DecodeK; };


// XYZZ (device) -> affine -> bytes; one thread per point
template <class F>
struct XyzzEncodeK {
  static constexpr int BLOCK = 32;
  PS_DEV static void run(uint32_t i, const XYZZ<F>* in, int format, uint8_t* out) {
    Affine<F> a = xyzz_to_affine_serial(in[i]);
    point_encode(a, format, out + (size_t)i * (format == PS_FMT_COMPRESSED ? PointBytes<F>::COMP : PointBytes<F>::AFF));
  }
};
template <class F>
struct AffineEncodeK {
  static constexpr int BLOCK = 128;
  PS_DEV static void run(uint32_t i, const Affine<F>* in, int format, uint8_t* out) {
    point_encode(in[i], format, out + (size_t)i * (format == PS_FMT_COMPRESSED ? PointBytes<F>::COMP : PointBytes<F>::AFF));
  }
};

}  // namespace ps
