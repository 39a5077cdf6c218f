// Test-only harness for the verifiers' arithmetic (tests/test_gpu_pairing.py, tests/test_host_pairing.py): the Fp6 / Fp12
// tower, the Frobenius map, the Miller loop and the final exponentiation of pairing.cuh, the pairing-product check, and
// the square roots, subgroup check and point decode / encode of codec.cuh -- value by value, not only verdicts.
//
// Raw Montgomery limbs go in and come out (Fp12 = 576 bytes: c0.{c0,c1,c2} then c1.{...}, each Fp2 c0 then c1, which is
// the oracle's tuple order); the Python side converts.  Compiled for sm_100a with the project's nvcc flags, every
// launcher runs on the legacy default stream, synchronises and returns the CUDA error code.  Compiled with
// g++ -x c++ -DPS_HOST_EMU (build.build_device_harness(host=True)) the same row bodies run in a serial loop on host
// pointers, so the CPU suite can check the same functions on a machine without a GPU.
#include "../playsnark_b200/csrc/codec.cuh"
#include "../playsnark_b200/csrc/pairing.cuh"

using namespace ps;

namespace {

// ---- row functors (one row per thread) -----------------------------------------------------------------------------
enum TowerOp {
  T_FP6_MUL = 0, T_FP6_INV, T_FP6_MUL_V, T_FP12_MUL, T_FP12_SQR, T_FP12_INV, T_FP12_CONJ, T_FP12_FROB, T_FP12_POW_X,
  T_FINAL_EXP,
};

template <int OP>
struct TowerK {
  // a, b: operands (Fp6 for the T_FP6_* ops, Fp12 otherwise); T_FP12_FROB applies fp12_frob k times
  PS_DEV static void run(uint32_t i, const void* a, const void* b, void* o, int k) {
    if constexpr (OP <= T_FP6_MUL_V) {
      const Fp6 x = static_cast<const Fp6*>(a)[i];
      Fp6 r;
      if constexpr (OP == T_FP6_MUL) r = fp6_mul(x, static_cast<const Fp6*>(b)[i]);
      else if constexpr (OP == T_FP6_INV) r = fp6_inv(x);
      else r = fp6_mul_v(x);
      static_cast<Fp6*>(o)[i] = r;
    } else {
      const Fp12 x = static_cast<const Fp12*>(a)[i];
      Fp12 r;
      if constexpr (OP == T_FP12_MUL) r = fp12_mul(x, static_cast<const Fp12*>(b)[i]);
      else if constexpr (OP == T_FP12_SQR) r = fp12_sqr(x);
      else if constexpr (OP == T_FP12_INV) r = fp12_inv(x);
      else if constexpr (OP == T_FP12_CONJ) r = fp12_conj(x);
      else if constexpr (OP == T_FP12_FROB) { r = x; for (int j = 0; j < k; j++) r = fp12_frob(r); }
      else if constexpr (OP == T_FP12_POW_X) r = fp12_pow_x(x);
      else r = final_exponentiation(x);
      static_cast<Fp12*>(o)[i] = r;
    }
  }
};

struct MillerK {
  PS_DEV static void run(uint32_t i, const G1Affine* P, const G2Affine* Q, Fp12* o) { o[i] = miller_loop(P[i], Q[i]); }
};

// the verdict of PairingCheckK itself, and the value it compares with one: the product of the check's Miller values
// taken in the same order, after the final exponentiation
struct CheckK {
  PS_DEV static void run(uint32_t t, const Fp12* f, const uint32_t* first, uint8_t* ok, Fp12* fe) {
    PairingCheckK::run(t, f, first, ok);
    Fp12 acc = Fp12::one();
    for (uint32_t i = first[t]; i < first[t + 1]; i++) acc = fp12_mul(acc, f[i]);
    fe[t] = final_exponentiation(acc);
  }
};

// square roots: o = the root codec.cuh returns, ok = whether it claims one
struct FpSqrtK {
  PS_DEV static void run(uint32_t i, const Fp* a, Fp* o, uint8_t* ok) { Fp r; ok[i] = fp_sqrt(a[i], r) ? 1 : 0; o[i] = r; }
};
struct Fp2SqrtK {
  PS_DEV static void run(uint32_t i, const Fp2* a, Fp2* o, uint8_t* ok) { Fp2 r; ok[i] = fp2_sqrt(a[i], r) ? 1 : 0; o[i] = r; }
};

template <class F>
struct SubgroupK {
  PS_DEV static void run(uint32_t i, const Affine<F>* p, uint8_t* ok) { ok[i] = in_subgroup(p[i]) ? 1 : 0; }
};

// k_i P_i over `nlimbs` little-endian limbs of k (8 per row in memory), returned affine
template <class F>
struct ScalarMulK {
  PS_DEV static void run(uint32_t i, const Affine<F>* p, const uint32_t* k, int nlimbs, Affine<F>* o) {
    o[i] = xyzz_to_affine_serial(xyzz_scalar_mul(XYZZ<F>::from_affine(p[i]), k + 8 * (size_t)i, nlimbs));
  }
};

// the decode kernels of the library with their per-point status byte (0 good, 2 bad encoding / off the curve, 4 outside
// the subgroup), then the decoded point encoded again in the same format
template <class F>
struct DecodeK {
  PS_DEV static void run(uint32_t i, const uint8_t* in, int format, int subgroup, Affine<F>* out, uint8_t* status,
                         uint8_t* again, uint32_t* err) {
    DecodeKernel<F>::K::run(i, in, format, out, err, subgroup, status);
    const size_t len = format == PS_FMT_COMPRESSED ? PointBytes<F>::COMP : PointBytes<F>::AFF;
    point_encode(out[i], format, again + i * len);
  }
};

// ---- launch --------------------------------------------------------------------------------------------------------
#if PS_GPU
template <class K, class... Args>
__global__ void dp_kernel(uint32_t n, Args... args) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) K::run(i, args...);
}
// 32 threads per block: every row is one long serial computation (Miller loop, exponentiation, scalar multiplication)
template <class K, class... Args>
int launch(int n, Args... args) {
  if (n <= 0) return 0;
  dp_kernel<K><<<(n + 31) / 32, 32>>>((uint32_t)n, args...);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  return (int)e;
}
#else
template <class K, class... Args>
int launch(int n, Args... args) {
  for (int i = 0; i < n; i++) K::run((uint32_t)i, args...);
  return 0;
}
#endif

}  // namespace

extern "C" {

// 1 = the CUDA build, 0 = the host build
int dp_is_device() { return PS_GPU; }

// op: TowerOp; k: the number of Frobenius applications for T_FP12_FROB; returns -1 for an unknown op
int dp_tower(int op, int k, const void* a, const void* b, void* o, int n) {
  switch (op) {
#define DP_T(OP) case OP: return launch<TowerK<OP>>(n, a, b, o, k);
    DP_T(T_FP6_MUL) DP_T(T_FP6_INV) DP_T(T_FP6_MUL_V) DP_T(T_FP12_MUL) DP_T(T_FP12_SQR) DP_T(T_FP12_INV) DP_T(T_FP12_CONJ)
    DP_T(T_FP12_FROB) DP_T(T_FP12_POW_X) DP_T(T_FINAL_EXP)
#undef DP_T
    default: return -1;
  }
}

int dp_miller(const void* P, const void* Q, void* o, int n) {
  return launch<MillerK>(n, (const G1Affine*)P, (const G2Affine*)Q, (Fp12*)o);
}

// checks t = 0 .. nchecks-1 over the Miller values [first[t], first[t+1])
int dp_check(const void* f, const uint32_t* first, uint8_t* ok, void* fe, int nchecks) {
  return launch<CheckK>(nchecks, (const Fp12*)f, first, ok, (Fp12*)fe);
}

// ext: 1 = Fp, 2 = Fp2
int dp_sqrt(int ext, const void* a, void* o, uint8_t* ok, int n) {
  if (ext == 1) return launch<FpSqrtK>(n, (const Fp*)a, (Fp*)o, ok);
  if (ext == 2) return launch<Fp2SqrtK>(n, (const Fp2*)a, (Fp2*)o, ok);
  return -1;
}

// group: 1 = G1, 2 = G2 (affine points, raw Montgomery limbs)
int dp_in_subgroup(int group, const void* p, uint8_t* ok, int n) {
  if (group == 1) return launch<SubgroupK<Fp>>(n, (const G1Affine*)p, ok);
  if (group == 2) return launch<SubgroupK<Fp2>>(n, (const G2Affine*)p, ok);
  return -1;
}

// k: 8 limbs per row, of which the low `nlimbs` (4 or 8) are used
int dp_scalar_mul(int group, int nlimbs, const void* p, const uint32_t* k, void* o, int n) {
  if (nlimbs != 4 && nlimbs != 8) return -1;
  if (group == 1) return launch<ScalarMulK<Fp>>(n, (const G1Affine*)p, k, nlimbs, (G1Affine*)o);
  if (group == 2) return launch<ScalarMulK<Fp2>>(n, (const G2Affine*)p, k, nlimbs, (G2Affine*)o);
  return -1;
}

// format: PS_FMT_COMPRESSED / PS_FMT_AFFINE; err: one word, OR-ed into (the caller zeroes it)
int dp_decode(int group, int format, int subgroup, const uint8_t* in, void* out, uint8_t* status, uint8_t* again,
              uint32_t* err, int n) {
  if (group == 1) return launch<DecodeK<Fp>>(n, in, format, subgroup, (G1Affine*)out, status, again, err);
  if (group == 2) return launch<DecodeK<Fp2>>(n, in, format, subgroup, (G2Affine*)out, status, again, err);
  return -1;
}

}  // extern "C"
