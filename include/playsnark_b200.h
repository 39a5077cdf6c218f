/* playsnark_b200 -- C ABI of the B200-native prover backend.
 *
 * Drop-in boundary for the proving path of nikkolasg/playsnark.  The reference has no FFI; its
 * boundary is the pair of Go functions
 *     Groth16Prove(tr Groth16Setup, q QAP, sol Vector) Groth16Proof      (groth16.go:122)
 *     PHGR13Prove(ek PHGR13EvalKey, qap QAP, solution Vector) PHGR13Proof (pinochio.go:207)
 * and the helpers they call (QAP.Quotient qap.go:151, Poly.BlindEval algebra.go:348).  A cgo shim
 * inside package playsnark marshals its kyber values with MarshalBinary and calls the entry points
 * below (INTEGRATION.md shows the shim).  Conventions:
 *   - every function returns an int status (PS_OK == 0); the shim maps PS_ERR_REMAINDER to
 *     panic("apocalypse") (qap.go:159, pinochio.go:215) and PS_ERR_LENGTH to the BlindEval length
 *     panic (algebra.go:350-352);
 *   - Fr scalars: 32 bytes, big-endian, canonical (< r)          (kyber Scalar.MarshalBinary);
 *   - G1 / G2 points: 48 / 96 bytes zcash-compressed (PS_FMT_COMPRESSED; kyber Point.MarshalBinary)
 *     or 96 / 192 bytes zcash-uncompressed (PS_FMT_AFFINE) for bulk keys already decompressed;
 *   - handles are opaque, caller-owned, freed with the matching *_free; buffers are caller-owned;
 *   - one ps_ctx per host thread and per GPU; no global state.
 * There is no CPU fallback: every entry point needs a CUDA device.
 */
#ifndef PLAYSNARK_B200_H
#define PLAYSNARK_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum {
  PS_OK = 0,
  PS_ERR_ARG = 1,        /* null pointer, bad size or bad enum */
  PS_ERR_LENGTH = 2,     /* len(p) != len(points): BlindEval's panic, algebra.go:350-352 */
  PS_ERR_REMAINDER = 3,  /* (a*b - c) mod z != 0: panic("apocalypse"), qap.go:158-160 */
  PS_ERR_ENCODING = 4,   /* point bytes do not decode to a curve point / scalar >= r */
  PS_ERR_CUDA = 5,
  PS_ERR_ALLOC = 6,
  PS_ERR_UNSUPPORTED = 7
};

enum { PS_FMT_COMPRESSED = 0, PS_FMT_AFFINE = 1 };
enum { PS_G1 = 1, PS_G2 = 2 };

typedef struct ps_ctx ps_ctx;
typedef struct ps_bases ps_bases;     /* resident MSM base set (G1 or G2)                      */
typedef struct ps_qap ps_qap;         /* resident QAP (dense polynomials or sparse R1CS)        */
typedef struct ps_g16_key ps_g16_key; /* resident Groth16 proving key                           */
typedef struct ps_phgr13_key ps_phgr13_key;

const char* ps_strerror(int status);
const char* ps_version(void);

/* ---- context ------------------------------------------------------------------------------ */
int ps_ctx_create(int device, ps_ctx** out);
/* run on a caller-provided CUDA stream (cudaStream_t passed as void*), e.g. torch's current one */
int ps_ctx_set_stream(ps_ctx* ctx, void* cuda_stream);
/* options: "subgroup_check" = 1 (points decoded by the loaders must lie in the prime-order subgroup, as kilic's
 * FromCompressed demands of the reference's keys; default) | 0 (skip the r-multiplication for vouched keys);
 * "msm_team" = 1 (latency-bound tail kernels of the MSM use a team of four lanes per group operation,
 * default) | 0 (one thread per operation);
 * "msm_shards" = N >= 1: base sets and keys loaded afterwards are meant to be summed in N index ranges
 * (one per GPU, ps_msm_device / ps_g16_msm_partials), so their automatic window is sized for n / N points;
 * "msm_bucket_cost" = cost of one bucket (merge + reduction) in the automatic window choice, in field
 * products with a mixed addition counting 10 (default 70, fitted on B200);
 * "msm_scatter" = 0 (one-pass counting sort of the bucket entries) | 1 (two-level sort, by partition of buckets and
 * then by bucket, from 2^25 entries n*W; default) | 2 (two-level sort whenever the bucket count allows; tests);
 * "msm_wave_floor" = 1 (short accumulate chunks: whole waves with the wave count rounded down, default) | 0 (rounded up);
 * "interp_fused" = 1 (lowest nine levels of the interpolation tree in one shared-memory kernel, default) | 0 (level by
 * level; identical coefficients).  Environment: PLAYSNARK_B200_STREAM2_PRIO=0 creates the secondary stream (G2 sums) at
 * default instead of high priority (A/B runs). */
int ps_ctx_set_option(ps_ctx* ctx, const char* name, int value);
int ps_ctx_sync(ps_ctx* ctx);
void ps_ctx_destroy(ps_ctx* ctx);
/* number of CUDA kernels this library has launched in this process (bench.py's gpu_launches) */
uint64_t ps_launch_count(void);

/* ---- MSM bases: the []Commit argument of Poly.BlindEval (algebra.go:348) ------------------- */
/* `window_bits` = 0 lets the library choose c per call; otherwise fixes the Pippenger window and,
 * with `precompute_tables` = T > 1, stores 2^(c*t) * P_i for t < T so that T windows share one
 * bucket set (T is clamped to the number of windows).  precompute_tables = -1 asks for all
 * windows, with the window chosen by the library when window_bits = 0 (what the key loaders use:
 * 180 GB of HBM make W copies of the key cheap, and they remove the per-window bucket sets).    */
int ps_bases_load(ps_ctx* ctx, int group, const uint8_t* points, size_t n, int format,
                  int window_bits, int precompute_tables, ps_bases** out);
size_t ps_bases_len(const ps_bases* b);
/* out[0] = window bits c used for a full-length MSM, out[1] = windows W, out[2] = tables T,
 * out[3] = group */
int ps_bases_info(const ps_bases* b, int out[4]);
void ps_bases_free(ps_bases* b);
/* bases[i] = scalars[i] * generator (GeneratePowersCommit's Mul(s, nil), algebra.go:373,381);
 * used by setup-side callers and the benchmarks to create large keys on the GPU.               */
int ps_bases_from_scalars(ps_ctx* ctx, int group, const uint8_t* scalars_be, size_t n,
                          int window_bits, int precompute_tables, ps_bases** out);
/* copy points [first, first+count) out as compressed or affine bytes */
int ps_bases_export(ps_ctx* ctx, const ps_bases* b, size_t first, size_t count, int format, uint8_t* out);

/* ---- MSM: Poly.BlindEval(zero, blindedPoint) = sum_i p[i] * P[i] (algebra.go:348-359) -------- */
/* n must equal ps_bases_len(b) (PS_ERR_LENGTH otherwise, like the reference's panic).
 * out: 48 B (G1) / 96 B (G2) compressed.                                                       */
int ps_msm(ps_ctx* ctx, const ps_bases* b, const uint8_t* scalars_be, size_t n, uint8_t* out);
/* `rows` MSMs against the same base set in one call (many BlindEvals against one resident key): scalars_be holds
 * rows x n scalars, row-major; out[k] = sum_i scalars[k][i] * P[i], `rows` compressed points.  n must equal
 * ps_bases_len(b) (PS_ERR_LENGTH otherwise).  All rows share one Pippenger pipeline (one bucket set per row), split
 * into several only when one pipeline would pass 2^31 bucket entries.  A base set loaded with all window tables
 * (precompute_tables = -1) is best given a window chosen for rows x n points and `rows` outputs.                  */
int ps_msm_rows(ps_ctx* ctx, const ps_bases* b, const uint8_t* scalars_be, size_t n, size_t rows, uint8_t* out);
/* Partial-range / device-resident variant for sharding and benchmarking: scalars already on the
 * device as 8 little-endian u32 limbs each, standard (non-Montgomery) form; sums bases
 * [first, first+n) and leaves the partial as an XYZZ point (4 field elements, Montgomery limbs)
 * in device memory `d_out_xyzz` (192 B G1 / 384 B G2).                                          */
int ps_msm_device(ps_ctx* ctx, const ps_bases* b, size_t first, const void* d_scalars_le, size_t n,
                  void* d_out_xyzz);
/* the same with the scalars in Montgomery form, as ps_fr_upload leaves them (host wire bytes -> device limbs) */
int ps_msm_device_mont(ps_ctx* ctx, const ps_bases* b, size_t first, const void* d_scalars_mont, size_t n,
                       void* d_out_xyzz);
/* sum `count` XYZZ partials (device memory, contiguous) and emit the compressed point: the single
 * small gather of the multi-GPU MSM.                                                            */
int ps_msm_combine(ps_ctx* ctx, int group, const void* d_partials_xyzz, size_t count, uint8_t* out);

/* ---- Fr polynomial kernels --------------------------------------------------------------------- */
/* in-place radix-2 NTT over Fr on `n = 2^log_n` big-endian scalars (host memory).  inverse != 0
 * computes the inverse transform (scaled by 1/n).  coset (32 B, may be NULL) evaluates on
 * coset * <omega> (forward) or interpolates from it (inverse).  omega = 7^((r-1)/2^log_n).      */
int ps_ntt_fr(ps_ctx* ctx, uint8_t* data_be, unsigned log_n, int inverse, const uint8_t* coset_be);

/* QAP as ToQAP produces it (qap.go:35-65): left/right/out are m polynomials of n coefficients
 * each (row-major m x n, 32 B big-endian, low degree first), z has n+1 coefficients.           */
int ps_qap_load_dense(ps_ctx* ctx, size_t n_gates, size_t n_vars, size_t n_io, const uint8_t* left,
                      const uint8_t* right, const uint8_t* out, const uint8_t* z, ps_qap** qap);
/* Sparse R1CS twin of the same object for sizes where the dense QAP cannot exist (3*m*n*32 B):
 * CSR matrices over the gates (row_ptr[n+1], col[nnz], val[nnz] as 32 B big-endian Fr); the
 * polynomials are implicit (interpolants on the domain {1..n}).  Any n_gates >= 2, like ToQAP.   */
int ps_qap_load_r1cs(ps_ctx* ctx, size_t n_gates, size_t n_vars, size_t n_io,
                     const uint32_t* l_row_ptr, const uint32_t* l_col, const uint8_t* l_val,
                     const uint32_t* r_row_ptr, const uint32_t* r_col, const uint8_t* r_val,
                     const uint32_t* o_row_ptr, const uint32_t* o_col, const uint8_t* o_val,
                     ps_qap** qap);
void ps_qap_free(ps_qap* qap);

/* QAP.Quotient (qap.go:151-162): witness = n_vars Fr values (Value.ToFieldElement, curve.go:17),
 * out_h = n_gates-1 coefficients.  PS_ERR_REMAINDER when z does not divide a*b-c.
 * out_abc (optional, may be NULL) receives computeAggregatePoly's three polynomials
 * (qap.go:164-175), 3 * n_gates * 32 B.                                                         */
int ps_quotient(ps_ctx* ctx, const ps_qap* qap, const uint8_t* witness_be, uint8_t* out_h, uint8_t* out_abc);

/* ---- Groth16 (groth16.go) ---------------------------------------------------------------------- */
/* Proving part of Groth16Setup (groth16.go:30-61): Xi[n], Xi2[n] (G2), XiT[n-1], NioLP[n_nio],
 * Alpha, Beta, Delta (G1), Beta2, Delta2 (G2).                                                   */
int ps_g16_key_load(ps_ctx* ctx, size_t n_gates, size_t n_nio, int format, const uint8_t* xi,
                    const uint8_t* xi2, const uint8_t* xit, const uint8_t* niolp, const uint8_t* alpha,
                    const uint8_t* beta, const uint8_t* delta, const uint8_t* beta2,
                    const uint8_t* delta2, ps_g16_key** key);
void ps_g16_key_free(ps_g16_key* key);
/* Groth16Prove (groth16.go:122-211) with the blinding scalars supplied by the caller (the shim
 * samples them with Pick(random.New()) as groth16.go:148,158 and stores them in the proof).
 * outA 48 B, outB 96 B, outC 48 B; out_h optional (n_gates-1 scalars).                          */
int ps_g16_prove(ps_ctx* ctx, const ps_g16_key* key, const ps_qap* qap, const uint8_t* witness_be,
                 const uint8_t* r_be, const uint8_t* s_be, uint8_t* outA, uint8_t* outB, uint8_t* outC,
                 uint8_t* out_h);

/* NewGroth16TrustedSetup (groth16.go:64-101, 238-264) on the device for a resident QAP, the toxic waste supplied by
 * the caller (the shim samples it with Pick(random.New()) and keeps it in Groth16Setup.tw): toxic_be = alpha, beta,
 * delta, x, gamma (5 x 32 B).  Produces the resident proving key; out_iolp ((n_vars - n_io) x 48 B, optional) and
 * out_gamma (96 B, optional) receive the verifier's IoLP and Gamma, compressed.  u_i(x), v_i(x), w_i(x) come from the
 * Lagrange basis at x (sparse QAP) or Horner (dense), the points from the fixed-base kernel.                       */
int ps_g16_setup(ps_ctx* ctx, const ps_qap* qap, const uint8_t* toxic_be, ps_g16_key** key, uint8_t* out_iolp,
                 uint8_t* out_gamma);
/* the elements of a resident key as wire bytes, to fill Groth16Setup's fields (any output may be NULL) */
int ps_g16_key_export(ps_ctx* ctx, const ps_g16_key* key, int format, uint8_t* xi, uint8_t* xi2, uint8_t* xit,
                      uint8_t* niolp, uint8_t* alpha, uint8_t* beta, uint8_t* delta, uint8_t* beta2, uint8_t* delta2);

/* Groth16 across several GPUs (one process per GPU, every process holds the key): rank 0 runs the
 * quotient and emits the scalar vectors of the proof's three MSMs (`which` 0 = A over G1, 1 = C over
 * G1, 2 = B over G2; standard-form limbs, 8 x u32 each, device memory sized by ps_g16_scalar_count);
 * after a broadcast every rank sums its index range with ps_msm_device over ps_g16_key_bases and the
 * partials are gathered and added with ps_msm_combine.                                           */
size_t ps_g16_scalar_count(const ps_g16_key* key, int which);
const ps_bases* ps_g16_key_bases(const ps_g16_key* key, int which);
int ps_g16_scalars(ps_ctx* ctx, const ps_g16_key* key, const ps_qap* qap, const uint8_t* witness_be,
                   const uint8_t* r_be, const uint8_t* s_be, void* d_scA, void* d_scC, void* d_scB);

/* the three partial MSMs of one rank in one call (G2 on the context's second stream):
 * first[i] / count[i] = index range of MSM i (0 = A, 1 = C, 2 = B) inside the key's base sets, scalar
 * pointers already offset to that range; d_partials receives [A 192 B | C 192 B | B 384 B] (XYZZ).    */
int ps_g16_msm_partials(ps_ctx* ctx, const ps_g16_key* key, const void* d_scA, const void* d_scC, const void* d_scB,
                        const size_t first[3], const size_t count[3], void* d_partials);
/* splitting the quotient over two GPUs (sparse QAP): ps_qap_aggregate_one interpolates one aggregate
 * polynomial (which = 0: a, 1: b; n Montgomery coefficients in device memory); after the exchange
 * ps_g16_scalars_from_ab does the gate check, the division and the scalar assembly.               */
int ps_qap_aggregate_one(ps_ctx* ctx, const ps_qap* qap, const uint8_t* witness_be, int which, void* d_out_coef);
int ps_g16_scalars_from_ab(ps_ctx* ctx, const ps_g16_key* key, const ps_qap* qap, const uint8_t* witness_be,
                           const uint8_t* r_be, const uint8_t* s_be, const void* d_a, const void* d_b,
                           void* d_scA, void* d_scC, void* d_scB);

/* Groth16 over 2 * parts GPUs (parts a power of two; sparse QAP), no host round trip between the
 * steps (errors are OR-ed into a device status word: bit 0 = scalar encoding, bit 1 = remainder, i.e.
 * the reference's "apocalypse" qap.go:159):
 *  Below np = the power of two >= max(n, 2): the leaves of the interpolation tree (gates above n are empty).
 *  - ps_qap_interp_part: rank (which, part) evaluates its np/parts gates (all three matrices, gate check
 *    a(j) b(j) = c(j) on them), and folds the subtree over those gates of polynomial `which` (0 = a,
 *    1 = b) up to one node: d_out_evals receives its 2 np/parts evaluations (Montgomery); with parts = 1
 *    it receives the n coefficients directly and no finish step is needed.  d_w_nio_out (optional)
 *    receives the last n_io witness values in standard form (head of C's scalar vector).
 *  - after an all-gather of the parts, ps_qap_interp_finish runs the top log2(parts) levels on the 2 np
 *    gathered evaluations and emits the n coefficients (Montgomery).
 *  - ps_g16_scalars_ab (every rank, from the broadcast a and b): scA = [a | r | 1], scB = [b | s | 1],
 *    scC_tail = [s a + r b | s | r | r s] (standard form; C's scalar vector is [w_nio | h | tail]), so
 *    that the MSMs A, B and the tail of C run while one rank divides;
 *  - ps_g16_h_from_ab: h = floor(a b / z), n - 1 standard-form values (to be broadcast into C's vector). */
int ps_qap_interp_part(ps_ctx* ctx, const ps_qap* qap, const uint8_t* witness_be, int which, size_t part,
                       size_t parts, void* d_out_evals, void* d_w_nio_out, void* d_status);
/* the same with the witness already on the device (n_vars Montgomery values), e.g. after every rank has
 * uploaded one slice with ps_fr_upload (host wire format -> Montgomery limbs in device memory, encoding
 * errors into the status word) and the slices have been all-gathered over NVLink: one upload of the
 * witness per node instead of one per GPU */
int ps_qap_interp_part_dev(ps_ctx* ctx, const ps_qap* qap, const void* d_witness_mont, int which, size_t part,
                           size_t parts, void* d_out_evals, void* d_w_nio_out, void* d_status);
int ps_fr_upload(ps_ctx* ctx, const uint8_t* values_be, size_t count, void* d_out_mont, void* d_status);
int ps_qap_interp_finish(ps_ctx* ctx, const ps_qap* qap, size_t parts, const void* d_evals_all, void* d_out_coef);
int ps_g16_scalars_ab(ps_ctx* ctx, const ps_g16_key* key, const uint8_t* r_be, const uint8_t* s_be, const void* d_a,
                      const void* d_b, void* d_scA, void* d_scB, void* d_scC_tail);
int ps_g16_h_from_ab(ps_ctx* ctx, const ps_qap* qap, const void* d_a, const void* d_b, void* d_h_out);
/* end of a sharded proof: `count` gathered records, `stride` bytes apart (a multiple of 16, >= 960), each
 * [A 192 B | C tail 192 B | B 384 B | C head 192 B | ...] as written by two ps_g16_msm_partials calls;
 * adds them up and emits the compressed proof elements (G2 on the second stream). */
int ps_g16_combine(ps_ctx* ctx, const void* d_records, size_t count, size_t stride, uint8_t* outA, uint8_t* outB,
                   uint8_t* outC);

/* Page-locked host memory for call arguments (witness, scalars): host-to-device copies from it run at
 * link speed and asynchronously; plain pageable buffers are accepted everywhere as well.          */
int ps_host_alloc(size_t bytes, void** out);
void ps_host_free(void* p);

/* ---- PHGR13 / Pinocchio (pinochio.go) ------------------------------------------------------------ */
/* PHGR13EvalKey (pinochio.go:37-62): gsi[n-1]; vs, ys, vas, was, yas, vbs, wbs, ybs [n_mid] in G1
 * (wbs is typed []G2 in the reference but holds G1 points, pinochio.go:114,136); ws [n_mid] G2. */
int ps_phgr13_key_load(ps_ctx* ctx, size_t n_gates, size_t n_mid, int format, const uint8_t* gsi,
                       const uint8_t* vs, const uint8_t* ws, const uint8_t* ys, const uint8_t* vas,
                       const uint8_t* was, const uint8_t* yas, const uint8_t* vbs, const uint8_t* wbs,
                       const uint8_t* ybs, ps_phgr13_key** key);
void ps_phgr13_key_free(ps_phgr13_key* key);
/* NewPHGR13TrustedSetup (pinochio.go:93-176) on the device: toxic_be = s, av, aw, ay, rv, rw, beta, gamma (8 x 32 B,
 * the reference's sampling order).  Produces the resident evaluation key and, on request, the verification key,
 * compressed: out_vk_fixed (576 B) = av (G2) | aw (G1) | ay (G2) | gamma (G2) | bgamma (G1) | bgamma2 (G2) | yts (G2);
 * out_vk_vs / _ws / _ys = the commitments of ALL n_vars variables (48 / 96 / 48 B each).                          */
int ps_phgr13_setup(ps_ctx* ctx, const ps_qap* qap, const uint8_t* toxic_be, ps_phgr13_key** key, uint8_t* out_vk_fixed,
                    uint8_t* out_vk_vs, uint8_t* out_vk_ws, uint8_t* out_vk_ys);
int ps_phgr13_key_export(ps_ctx* ctx, const ps_phgr13_key* key, int format, uint8_t* gsi, uint8_t* vs, uint8_t* ws,
                         uint8_t* ys, uint8_t* vas, uint8_t* was, uint8_t* yas, uint8_t* vbs, uint8_t* wbs, uint8_t* ybs);
/* ---- verifiers (SURVEY 8 f4) -----------------------------------------------------------------------------------
 * The reference compares GT values for equality only; every such equation is decided as prod_i e(P_i, Q_i) == 1.
 * ps_pairing_check_batch: n_checks independent products; check t covers counts[t] consecutive pairs of the flat point
 * arrays (wire format `format`); ok[t] = 1 when its product is 1.  One thread per Miller loop and per final
 * exponentiation: the parallelism is across pairs, checks and the proofs of a batch.  Points are validated like key
 * material (curve, subgroup): PS_ERR_ENCODING otherwise.  Replaces Suite.Pair + Equal, curve.go:36-38.           */
int ps_pairing_check_batch(ps_ctx* ctx, const uint8_t* g1_points, const uint8_t* g2_points, const uint32_t* counts,
                           size_t n_checks, int format, uint8_t* ok);
/* Groth16Verify (groth16.go:214-233): e(A, B) == e(Alpha, Beta2) e(sum_i io[i] IoLP[i], Gamma) e(C, Delta2).
 * Compressed points; iolp = n_io points of 48 B, io_be = n_io scalars (32 B big-endian); *ok = 1 / 0.             */
int ps_g16_verify(ps_ctx* ctx, const uint8_t* alpha, const uint8_t* beta2, const uint8_t* gamma2, const uint8_t* delta2,
                  const uint8_t* iolp, size_t n_io, const uint8_t* io_be, const uint8_t* A, const uint8_t* B,
                  const uint8_t* C, int* ok);
/* Groth16Verify for n_proofs proofs against one key as ONE combined pairing-product check with random 128-bit weights
 * rho_i:  prod_i e(-rho_i A_i, B_i) e(S Alpha, Beta2) e(L, Gamma) e(Cs, Delta2) == 1  with S = sum rho_i,
 * L = sum_j (sum_i rho_i io_i[j]) IoLP_j (one MSM), Cs = sum rho_i C_i: n_proofs + 3 Miller loops, one final exponentiation.
 * A batch of valid proofs is accepted; one with an invalid proof is rejected except with probability <= 2^-128 over the
 * weights, which must therefore be unpredictable to whoever made the proofs.
 *   io_be: n_proofs x n_io x 32 bytes, proof-major.  A / B / C: n_proofs compressed points each (48 / 96 / 48 B).
 *   weights: NULL (drawn by the library from the operating system: getrandom) or n_proofs x 16 bytes big-endian (tests).
 *   *ok = 1 iff every proof verifies.  per_proof: NULL, or n_proofs bytes, 1 = that proof verifies (on a failed batch the
 *   library bisects over a binary tree of the proofs: O(k log n_proofs) node checks for k invalid proofs).
 * Status:
 *   - a key point that does not decode (curve; subgroup when the "subgroup_check" option is set): PS_ERR_ENCODING;
 *     an io value >= r: PS_ERR_ENCODING;
 *   - a proof point that does not decode or lies outside the prime-order subgroup (always checked, whatever
 *     "subgroup_check" says): that proof is invalid (per_proof[i] = 0, *ok = 0) and left out of the combined sums; the
 *     call returns PS_OK and decides the other proofs;
 *   - a weight of zero: PS_ERR_ARG;  n_proofs == 0: *ok = 1, nothing launched;
 *   - n_proofs > 2^20, or n_proofs * n_io >= 2^31: PS_ERR_UNSUPPORTED.                                                */
int ps_g16_verify_batch(ps_ctx* ctx, const uint8_t* alpha, const uint8_t* beta2, const uint8_t* gamma2,
                        const uint8_t* delta2, const uint8_t* iolp, size_t n_io, size_t n_proofs, const uint8_t* io_be,
                        const uint8_t* A, const uint8_t* B, const uint8_t* C, const uint8_t* weights,
                        int* ok, uint8_t* per_proof);
/* PHGR13Verify (pinochio.go:281-375): division check, three CRS checks, linear check.  vk_fixed = the 576 bytes of
 * ps_phgr13_setup; vs / ws / ys = the commitments of the first n_io (public) variables (48 / 96 / 48 B each);
 * proof = the 432 bytes of ps_phgr13_prove.                                                                     */
int ps_phgr13_verify(ps_ctx* ctx, const uint8_t* vk_fixed, const uint8_t* vs, const uint8_t* ws, const uint8_t* ys,
                     size_t n_io, const uint8_t* io_be, const uint8_t* proof, int* ok);
/* PHGR13Verify for n_proofs proofs against one key as ONE combined pairing-product check.  Proof i gets five independent
 * random nonzero 128-bit weights rho_i1..rho_i5, one per equation of pinochio.go:312-372, and the batch is accepted iff
 *   prod_i e(rho1 gv_i, gw_i) * e(sum_i [rho2 vass_i + rho3 wass_i + rho4 yass_i - rho1 yss_i]
 *                                 - sum_k (sum_i rho_i1 io_ik) ys_k, G2gen)
 *   * e(-sum rho1 hs_i, yts) e(-sum rho2 vss_i, av) e(-sum rho4 yss_i, ay) e(sum rho5 gz_i, gamma)
 *   * e(-sum rho5 (vss_i + yss_i), bgamma2) e(-aw, sum rho3 wss_i) e(-bgamma, sum rho5 wss_i) == 1
 * with gv_i = sum_k io_ik vs_k + vss_i and gw_i = sum_k io_ik ws_k + wss_i: n_proofs + 8 Miller loops and one final
 * exponentiation.  A batch with an invalid proof is accepted with probability <= 2^-128 over the weights.
 *   vk_fixed, vs, ws, ys, n_io: as ps_phgr13_verify.  io_be: n_proofs x n_io x 32 bytes, proof-major.
 *   proofs: n_proofs x 432 bytes, each in ps_phgr13_prove's order.
 *   weights: NULL (drawn by the library: getrandom) or n_proofs x 5 x 16 bytes big-endian (tests).
 *   *ok, per_proof, and the status codes: as ps_g16_verify_batch (all 8 points of every proof are checked for the
 *   curve and the subgroup; a proof that fails is invalid and left out of the sums).                              */
int ps_phgr13_verify_batch(ps_ctx* ctx, const uint8_t* vk_fixed, const uint8_t* vs, const uint8_t* ws, const uint8_t* ys,
                           size_t n_io, size_t n_proofs, const uint8_t* io_be, const uint8_t* proofs,
                           const uint8_t* weights, int* ok, uint8_t* per_proof);

/* PHGR13Prove (pinochio.go:207-254).  out: hs, vss, yss, vass, wass, yass, gz (7 x 48 B, in this
 * order) then wss (96 B) = 432 bytes.                                                           */
int ps_phgr13_prove(ps_ctx* ctx, const ps_phgr13_key* key, const ps_qap* qap, const uint8_t* witness_be,
                    uint8_t* out432, uint8_t* out_h);

/* ---- several GPUs behind ONE call ------------------------------------------------------------------------------
 * A ps_mctx owns one context and one worker thread per listed device of this box.  A multi-GPU call does the
 * whole choreography inside the library: the devices exchange data over NVLink peer memory (no NCCL, no second
 * process), so a Go caller of Groth16Prove (groth16.go:122) makes exactly one cgo call per proof.
 * Keys are SHARDED: each device holds its index ranges of Xi, Xi2, XiT, NioLP (with all window tables); the
 * sparse QAP is replicated.  ps_mctx_set_option forwards ps_ctx options to every device; in addition
 * "rank0_share_percent" = MSM share of device 0 relative to the others (it also divides; 0 = automatic).   */
typedef struct ps_mctx ps_mctx;
typedef struct ps_mbases ps_mbases;
typedef struct ps_mqap ps_mqap;
typedef struct ps_mg16_key ps_mg16_key;
int ps_mctx_create(const int* devices, int ndev, ps_mctx** out);
void ps_mctx_destroy(ps_mctx* m);
int ps_mctx_size(const ps_mctx* m);
ps_ctx* ps_mctx_ctx(ps_mctx* m, int i);           /* the context of device i, for single-device calls */
int ps_mctx_set_option(ps_mctx* m, const char* name, int value);
/* MSM with the bases sharded by point range (SURVEY 8 e1): every device sums its range, the partial points are
 * pushed to device 0 and added there.  Same contract as ps_bases_load / ps_bases_from_scalars / ps_msm.     */
int ps_mbases_load(ps_mctx* m, int group, const uint8_t* points, size_t n, int format, int window_bits,
                   int precompute_tables, ps_mbases** out);
int ps_mbases_from_scalars(ps_mctx* m, int group, const uint8_t* scalars_be, size_t n, int window_bits,
                           int precompute_tables, ps_mbases** out);
size_t ps_mbases_len(const ps_mbases* b);
void ps_mbases_free(ps_mbases* b);
int ps_mmsm(ps_mctx* m, const ps_mbases* b, const uint8_t* scalars_be, size_t n, uint8_t* out);
/* Groth16: same arguments as ps_g16_key_load / ps_qap_load_r1cs / ps_qap_load_dense / ps_g16_prove.
 * With 2 * 2^j devices and a sparse QAP the whole proof is pipelined over the devices (interpolation split by
 * subtree, MSM shards overlapped with the division); otherwise device 0 runs the quotient and every device
 * its MSM shards.                                                                                           */
int ps_mg16_key_load(ps_mctx* m, size_t n_gates, size_t n_nio, int format, const uint8_t* xi, const uint8_t* xi2,
                     const uint8_t* xit, const uint8_t* niolp, const uint8_t* alpha, const uint8_t* beta,
                     const uint8_t* delta, const uint8_t* beta2, const uint8_t* delta2, ps_mg16_key** key);
void ps_mg16_key_free(ps_mg16_key* key);
int ps_mqap_load_r1cs(ps_mctx* m, size_t n_gates, size_t n_vars, size_t n_io,
                      const uint32_t* l_row_ptr, const uint32_t* l_col, const uint8_t* l_val,
                      const uint32_t* r_row_ptr, const uint32_t* r_col, const uint8_t* r_val,
                      const uint32_t* o_row_ptr, const uint32_t* o_col, const uint8_t* o_val, ps_mqap** qap);
int ps_mqap_load_dense(ps_mctx* m, size_t n_gates, size_t n_vars, size_t n_io, const uint8_t* left,
                       const uint8_t* right, const uint8_t* out, const uint8_t* z, ps_mqap** qap);
void ps_mqap_free(ps_mqap* qap);
int ps_mg16_prove(ps_mctx* m, const ps_mg16_key* key, const ps_mqap* qap, const uint8_t* witness_be,
                  const uint8_t* r_be, const uint8_t* s_be, uint8_t* outA, uint8_t* outB, uint8_t* outC);
/* stage marks of the last ps_mg16_prove on device `dev` (CUDA events on its stream): out_ms[k] = ms from the
 * start of the call's device work to mark k + 1; *count = values written                                    */
int ps_mg16_last_timeline(ps_mctx* m, int dev, float* out_ms, int max, int* count);

/* ---- measurement helpers (bench.py) ---------------------------------------------------------------- */
/* Integer-multiply pipe microbenchmark: variant 0 = IMAD (mad.lo), 1 = IMAD.HI, 2 = IMAD.WIDE
 * (independent), 3 = IMAD.WIDE.X carry chains as in the field multiplier; returns instructions/s
 * over all SMs measured with CUDA events.                                                       */
int ps_bench_intpipe(ps_ctx* ctx, int variant, int iters, double* inst_per_s, double* ms);
/* chained Montgomery products per second (field 0 = Fr, 1 = Fp) */
int ps_bench_fieldmul(ps_ctx* ctx, int field, int iters, double* mul_per_s, double* ms);
/* device time in ms of the last MSM on this context (CUDA events on its stream), by phase:
 * [0] digits+sort, [1] bucket-accumulate kernel, [2] partial merge, [3] bucket reduce, [4] total */
int ps_last_msm_timing(ps_ctx* ctx, float out_ms[5]);
/* device time in ms of the last ps_g16_prove: [0] quotient (aggregate / interpolation / NTT division),
 * [1] MSMs A and C (G1, one batched pipeline), [2] 0 (kept for layout), [3] normalise + encode A and C, [4] what
 * then remains of MSM B and its encoding (G2, concurrently on a second stream), [5] total          */
int ps_last_prove_timing(ps_ctx* ctx, float out_ms[6]);
/* device time in ms of the last batch verifier call (ps_g16_verify_batch or ps_phgr13_verify_batch), by phase:
 * [0] upload of points and weights, [1] decode + subgroup checks, [2] weighting (Groth16: rho_i A_i, rho_i C_i;
 * PHGR13: the weighted proof points), [3] upload + conversion of the io values (PHGR13: also the per-proof io MSMs
 * of gv_i in G1 and gw_i in G2), [4] the proofs' Miller loops, [5] tree of products and sums, [6] root check (io sums
 * + MSM, the fixed pairs' Miller loops, final exponentiation), [7] bisection for the per-proof verdicts, [8] total  */
int ps_last_verify_batch_timing(ps_ctx* ctx, float out_ms[9]);

#ifdef __cplusplus
}
#endif
#endif /* PLAYSNARK_B200_H */
