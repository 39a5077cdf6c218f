// Test-only device harness for the field and group arithmetic the kernels run (tests/test_gpu_arith.py).
//
// The host build of the same templates (tests/host_check.cpp) emulates the carry flag; this file compiles them for
// sm_100a with the project's nvcc flags, so the PTX carry chains (add.cc / madc), the inlined Fp2 tower of the G2 hot
// loop and the lane-cooperative group law of team.cuh (device-only) are what is checked.  Three kinds of kernels:
//   da_fe / da_fp2       element-wise operations on operands given by the caller, checked in Python against integers;
//   da_diff              one quantity computed by two independent routes on operands generated in the kernel from a
//                        counter-based hash (every limb saturating), for row counts Python cannot check;
//   da_group             serial and team group law on points given by the caller, checked against the oracle.
// Every launcher runs on the legacy default stream, synchronises and returns the CUDA error code.
#include "../playsnark_b200/csrc/team.cuh"
#include <cuda_runtime.h>

using namespace ps;

namespace {

template <class T>
__device__ __forceinline__ T ld(const uint32_t* p, size_t i) {
  T r;
  uint32_t* d = reinterpret_cast<uint32_t*>(&r);
#pragma unroll
  for (int k = 0; k < (int)(sizeof(T) / 4); k++) d[k] = p[i * (sizeof(T) / 4) + k];
  return r;
}
template <class T>
__device__ __forceinline__ void st(uint32_t* p, size_t i, const T& v) {
  const uint32_t* s = reinterpret_cast<const uint32_t*>(&v);
#pragma unroll
  for (int k = 0; k < (int)(sizeof(T) / 4); k++) p[i * (sizeof(T) / 4) + k] = s[k];
}

// ---- element-wise ------------------------------------------------------------------------------------------------
// Operation codes shared with tests/test_gpu_arith.py.  `std`: operands are plain integers, converted with to_mont on
// load and from_mont on store (as tests/host_check.cpp does); otherwise the raw limbs go in and come out unchanged.
enum FeOp {
  FE_MUL = 0, FE_ADD, FE_SUB, FE_SQR, FE_NEG, FE_FROM_MONT, FE_TO_MONT, FE_INV, FE_INV_SERIAL,
  FE_MUL_WIDE = 10, FE_MUL2_WIDE, FE_REDC_WIDE, FE_MUL2_LAZY, FE_SQRT, FE_NEG_LAZY,
};

template <class P, int OP>
__global__ void k_fe(const uint32_t* a, const uint32_t* b, const uint32_t* c, const uint32_t* d, uint32_t* o, int n, int std_) {
  using F = Fe<P>;
  constexpr int N = P::N;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if constexpr (OP == FE_MUL_WIDE || OP == FE_MUL2_WIDE) {   // plain 2N-limb integers a b (+ c d)
    uint32_t T[2 * N];
    if constexpr (OP == FE_MUL_WIDE) mul_wide(T, ld<F>(a, i), ld<F>(b, i));
    else mul2_wide(T, ld<F>(a, i), ld<F>(b, i), ld<F>(c, i), ld<F>(d, i));
#pragma unroll
    for (int k = 0; k < 2 * N; k++) o[(size_t)i * 2 * N + k] = T[k];
  } else if constexpr (OP == FE_REDC_WIDE) {                  // a holds 2N limbs
    uint32_t T[2 * N];
#pragma unroll
    for (int k = 0; k < 2 * N; k++) T[k] = a[(size_t)i * 2 * N + k];
    st(o, i, redc_wide<P>(T));
  } else if constexpr (OP == FE_MUL2_LAZY) {                  // (a b - c d) / R, the Y3 of every curve formula
    st(o, i, mul2_lazy(ld<F>(a, i), ld<F>(b, i), neg_lazy(ld<F>(c, i)), ld<F>(d, i)));
  } else if constexpr (OP == FE_NEG_LAZY) {
    st(o, i, neg_lazy(ld<F>(a, i)));
  } else {
    F x = ld<F>(a, i), y = ld<F>(b, i), r;
    if (std_) { x = x.to_mont(); y = y.to_mont(); }
    if constexpr (OP == FE_MUL) r = x * y;
    else if constexpr (OP == FE_ADD) r = x + y;
    else if constexpr (OP == FE_SUB) r = x - y;
    else if constexpr (OP == FE_SQR) r = x.sqr();
    else if constexpr (OP == FE_NEG) r = x.neg();
    else if constexpr (OP == FE_FROM_MONT) r = x.from_mont();
    else if constexpr (OP == FE_TO_MONT) r = x.to_mont();
    else if constexpr (OP == FE_INV) { if constexpr (N == 12) r = fp_inv(x); else r = fr_inv(x); }
    else if constexpr (OP == FE_INV_SERIAL) { if constexpr (N == 12) r = fp_inv_serial(x); else r = fr_inv_serial(x); }
    else if constexpr (OP == FE_SQRT) r = fp_sqrt_candidate(x);
    if (std_) r = r.from_mont();
    st(o, i, r);
  }
}

enum Fp2Op { F2_MUL = 0, F2_SQR, F2_INV, F2_INV_SERIAL };

// always plain integers in and out (c0, c1 of 12 limbs each)
template <bool I, int OP>
__global__ void k_fp2(const uint32_t* a, const uint32_t* b, uint32_t* o, int n) {
  using F = Fp2T<I>;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  F x = ld<F>(a, i), y = ld<F>(b, i), r;
  x = F{x.c0.to_mont(), x.c1.to_mont()};
  y = F{y.c0.to_mont(), y.c1.to_mont()};
  if constexpr (OP == F2_MUL) r = x * y;
  else if constexpr (OP == F2_SQR) r = x.sqr();
  else if constexpr (OP == F2_INV) r = FieldInv<F>::inv(x);
  else r = FieldInv<F>::inv_serial(x);
  st(o, i, F{r.c0.from_mont(), r.c1.from_mont()});
}

// ---- differential ------------------------------------------------------------------------------------------------
// Limb k of operand j of row r: SAT[h % 7] with h = mix(seed ^ mix(r * 64 + j * 16 + k)) (splitmix64's finaliser);
// the top limb is masked to the largest 2^m - 1 below the modulus' top limb, so every value is a field element.
__device__ __forceinline__ uint64_t mix64(uint64_t z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
__constant__ uint32_t c_SAT[7] = {0u, 1u, 2u, 0x7FFFFFFFu, 0x80000000u, 0xFFFFFFFEu, 0xFFFFFFFFu};

template <class P>
__device__ Fe<P> gen_sat(uint64_t seed, uint64_t row, int j) {
  constexpr int N = P::N;
  uint32_t top = P::MOD(N - 1), mask = 0xFFFFFFFFu;
  while (mask >= top) mask >>= 1;
  Fe<P> r;
#pragma unroll
  for (int k = 0; k < N; k++) r.v[k] = c_SAT[mix64(seed ^ mix64(row * 64 + j * 16 + k)) % 7];
  r.v[N - 1] &= mask;
  return r;
}

enum DiffOp { D_MUL2_LAZY = 0, D_REDC_WIDE, D_FP2_INLINE };

template <int OP>
__global__ void k_diff(uint64_t seed, uint64_t rows, unsigned long long* nbad, unsigned long long* bad_rows, int max_bad) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += stride) {
    bool ok;
    if constexpr (OP == D_MUL2_LAZY) {     // one reduction of a b + (p - c) d  vs  two reduced products
      Fp a = gen_sat<FpParams>(seed, r, 0), b = gen_sat<FpParams>(seed, r, 1);
      Fp c = gen_sat<FpParams>(seed, r, 2), d = gen_sat<FpParams>(seed, r, 3);
      ok = mul2_lazy(a, b, neg_lazy(c), d) == a * b - c * d;
    } else if constexpr (OP == D_REDC_WIDE) {   // Montgomery product vs plain product + separate reduction
      Fp a = gen_sat<FpParams>(seed, r, 0), b = gen_sat<FpParams>(seed, r, 1);
      uint32_t T[24];
      mul_wide(T, a, b);
      ok = a * b == redc_wide<FpParams>(T);
    } else {                                     // inlined vs out-of-line Fp2 tower, product and square
      Fp2 x{gen_sat<FpParams>(seed, r, 0), gen_sat<FpParams>(seed, r, 1)};
      Fp2 y{gen_sat<FpParams>(seed, r, 2), gen_sat<FpParams>(seed, r, 3)};
      Fp2I xi{x.c0, x.c1}, yi{y.c0, y.c1};
      Fp2 m = x * y, s = x.sqr();
      Fp2I mi = xi * yi, si = xi.sqr();
      ok = m.c0 == mi.c0 && m.c1 == mi.c1 && s.c0 == si.c0 && s.c1 == si.c1;
    }
    if (!ok) {
      unsigned long long k = atomicAdd(nbad, 1ull);
      if (k < (unsigned long long)max_bad) bad_rows[k] = r;
    }
  }
}

// ---- group law ---------------------------------------------------------------------------------------------------
// Operands: acc (XYZZ) and q (XYZZ for add, affine for madd, unused for doublings), raw Montgomery limbs.  Serial
// kernels write one XYZZ per item; team kernels run four lanes per item and every lane writes the point it holds
// (out[4 i + lane]), so the caller also sees that the lanes of a team agree.
enum GroupOp { G_MADD = 0, G_ADD, G_DBL, G_ADD_TEAM, G_DBL_TEAM };

template <class F, int OP>
__global__ void k_group(const uint32_t* acc, const uint32_t* q, uint32_t* out, int n) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if constexpr (OP == G_ADD_TEAM || OP == G_DBL_TEAM) {
    const TeamCtx tc = TeamCtx::of(t);
    const uint32_t i = t >> 2;
    if (i >= (uint32_t)n) return;   // all four lanes of a team leave together
    XYZZ<F> a = ld<XYZZ<F>>(acc, i);
    if constexpr (OP == G_ADD_TEAM) xyzz_add_t(a, ld<XYZZ<F>>(q, i), tc);
    else xyzz_dbl_t(a, tc);
    st(out, t, a);
  } else {
    if (t >= (uint32_t)n) return;
    XYZZ<F> a = ld<XYZZ<F>>(acc, t);
    if constexpr (OP == G_MADD) xyzz_madd(a, ld<Affine<F>>(q, t));
    else if constexpr (OP == G_ADD) xyzz_add(a, ld<XYZZ<F>>(q, t));
    else a = xyzz_dbl(a);
    st(out, t, a);
  }
}

int finish() {
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  return (int)e;
}
constexpr int BLK = 128;
inline int blocks(long long threads) { return (int)((threads + BLK - 1) / BLK); }

}  // namespace

extern "C" {

// field: 0 = Fp, 1 = Fr (FE_MUL_WIDE .. FE_NEG_LAZY: Fp only); returns -1 for an unknown combination
int da_fe(int field, int op, int std_, const uint32_t* a, const uint32_t* b, const uint32_t* c, const uint32_t* d, uint32_t* o, int n) {
  if (n <= 0) return 0;
#define DA_FE(P, OP) case OP: k_fe<P, OP><<<blocks(n), BLK>>>(a, b, c, d, o, n, std_); break;
  if (field == 0) {
    switch (op) {
      DA_FE(FpParams, FE_MUL) DA_FE(FpParams, FE_ADD) DA_FE(FpParams, FE_SUB) DA_FE(FpParams, FE_SQR)
      DA_FE(FpParams, FE_NEG) DA_FE(FpParams, FE_FROM_MONT) DA_FE(FpParams, FE_TO_MONT) DA_FE(FpParams, FE_INV)
      DA_FE(FpParams, FE_INV_SERIAL) DA_FE(FpParams, FE_MUL_WIDE) DA_FE(FpParams, FE_MUL2_WIDE)
      DA_FE(FpParams, FE_REDC_WIDE) DA_FE(FpParams, FE_MUL2_LAZY) DA_FE(FpParams, FE_SQRT) DA_FE(FpParams, FE_NEG_LAZY)
      default: return -1;
    }
  } else if (field == 1) {
    switch (op) {
      DA_FE(FrParams, FE_MUL) DA_FE(FrParams, FE_ADD) DA_FE(FrParams, FE_SUB) DA_FE(FrParams, FE_SQR)
      DA_FE(FrParams, FE_NEG) DA_FE(FrParams, FE_FROM_MONT) DA_FE(FrParams, FE_TO_MONT) DA_FE(FrParams, FE_INV)
      DA_FE(FrParams, FE_INV_SERIAL)
      default: return -1;
    }
  } else {
    return -1;
  }
#undef DA_FE
  return finish();
}

// inlined: 0 = Fp2 (out-of-line base-field products), 1 = Fp2I (inlined); F2_INV_SERIAL for both
int da_fp2(int inlined, int op, const uint32_t* a, const uint32_t* b, uint32_t* o, int n) {
  if (n <= 0) return 0;
#define DA_F2(I, OP) case OP: k_fp2<I, OP><<<blocks(n), BLK>>>(a, b, o, n); break;
  if (inlined) {
    switch (op) { DA_F2(true, F2_MUL) DA_F2(true, F2_SQR) DA_F2(true, F2_INV) DA_F2(true, F2_INV_SERIAL) default: return -1; }
  } else {
    switch (op) { DA_F2(false, F2_MUL) DA_F2(false, F2_SQR) DA_F2(false, F2_INV) DA_F2(false, F2_INV_SERIAL) default: return -1; }
  }
#undef DA_F2
  return finish();
}

// counts the rows of [0, rows) where the two routes disagree into *nbad (zeroed here); the first max_bad such rows
// (in no particular order) go to bad_rows
int da_diff(int op, unsigned long long seed, unsigned long long rows, unsigned long long* nbad, unsigned long long* bad_rows, int max_bad) {
  if (cudaMemset(nbad, 0, sizeof(unsigned long long)) != cudaSuccess) return finish();
  int sms = 0;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
  const int grid = (sms > 0 ? sms : 148) * 16;
  switch (op) {
    case D_MUL2_LAZY: k_diff<D_MUL2_LAZY><<<grid, 256>>>(seed, rows, nbad, bad_rows, max_bad); break;
    case D_REDC_WIDE: k_diff<D_REDC_WIDE><<<grid, 256>>>(seed, rows, nbad, bad_rows, max_bad); break;
    case D_FP2_INLINE: k_diff<D_FP2_INLINE><<<grid, 256>>>(seed, rows, nbad, bad_rows, max_bad); break;
    default: return -1;
  }
  return finish();
}

// group: 1 = G1 (Fp), 2 = G2 (Fp2), 3 = G2 over Fp2I (the type of the G2 bucket-accumulation kernel; madd only)
int da_group(int group, int op, const uint32_t* acc, const uint32_t* q, uint32_t* out, int n) {
  if (n <= 0) return 0;
  const long long threads = (op == G_ADD_TEAM || op == G_DBL_TEAM) ? 4LL * n : n;
#define DA_G(F, OP) case OP: k_group<F, OP><<<blocks(threads), BLK>>>(acc, q, out, n); break;
  if (group == 1) {
    switch (op) { DA_G(Fp, G_MADD) DA_G(Fp, G_ADD) DA_G(Fp, G_DBL) DA_G(Fp, G_ADD_TEAM) DA_G(Fp, G_DBL_TEAM) default: return -1; }
  } else if (group == 2) {
    switch (op) { DA_G(Fp2, G_MADD) DA_G(Fp2, G_ADD) DA_G(Fp2, G_DBL) DA_G(Fp2, G_ADD_TEAM) DA_G(Fp2, G_DBL_TEAM) default: return -1; }
  } else if (group == 3) {
    switch (op) { DA_G(Fp2I, G_MADD) default: return -1; }
  } else {
    return -1;
  }
#undef DA_G
  return finish();
}

}  // extern "C"
