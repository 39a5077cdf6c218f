// Per-group (G1 / G2) device operations behind the C ABI, declared once and instantiated in their own
// translation units (group_g1.cu, group_g2.cu) so that the orchestration code in capi.cu compiles in
// seconds and a change to one group's kernels rebuilds one object file.
//   GroupOps<Fp>  = G1 over Fp,  GroupOps<Fp2> = G2 over Fp2 = Fp[u]/(u^2+1)
#pragma once
#include "context.cuh"
#include "curve.cuh"

#ifndef PS_BUCKET_COST
#define PS_BUCKET_COST 70   // see msm_pick_window_full
#endif

namespace ps {

// A call runs a BATCH of multi-scalar multiplications through one pipeline: up to MSM_MAX_SEG segments
// (a run of scalars against one index range of one base set) feeding up to MSM_MAX_SEG outputs ("sets"
// of buckets, one per base set / result point).  All of them share the window geometry, so the digit
// pass, the sort, the bucket accumulation and above all the latency-bound merge / reduction tail run
// once for the whole batch: PHGR13's five sums over the same scalars (pinochio.go:231-241), Groth16's A
// and C, or the pieces of a sharded proof cost one tail instead of one each.
constexpr int MSM_MAX_SEG = 12;
struct MsmSeg {
  const uint32_t* scalars;  // n x 8 little-endian limbs
  uint32_t n;               // scalars / points of this segment
  uint32_t start;           // index of its first scalar in the batch's flat numbering
  uint32_t first;           // first point of the range inside each table of its base set
  uint32_t set;             // output slot (and base set) it accumulates into
  uint32_t mont;            // scalars are in Montgomery form
};
struct MsmPlan {
  int c;           // window bits
  int W;           // windows = ceil(255 / c)
  int T;           // precomputed tables per base set
  int S;           // bucket sets per output = ceil(W / T)
  uint32_t D;      // buckets per set = 2^(c-1)
  uint32_t total;  // scalars in the batch
  int nseg, nsets;
  // 0: segment mode (above).  Otherwise ROW mode: many MSMs of row_len scalars each against the same points of one base
  // set -- seg[0] holds the scalars of all rows, contiguous and row-major; scalar i goes to output i / row_len and point
  // seg[0].first + i % row_len; nbase[0] / toff[0] describe the base set; nsets = rows, not bounded by MSM_MAX_SEG
  uint32_t row_len;
  MsmSeg seg[MSM_MAX_SEG];
  uint32_t nbase[MSM_MAX_SEG];  // per output: points per table (table stride)
  uint32_t toff[MSM_MAX_SEG];   // per output: offset (in points) of its first table inside the slab all outputs share
};
inline int msm_windows(int c) { return (255 + c - 1) / c; }

// cost model (field multiplications) used to pick c when the bases carry no precomputed tables
inline int msm_pick_window(size_t n) {
  int best = 4; double best_cost = 1e300;
  for (int c = 4; c <= 22; c++) {
    double W = msm_windows(c);
    double buckets = W * (double)(1u << (c - 1));
    double cost = (double)n * W * 10.0 + buckets * (2.0 * 14.0 + 10.0);
    if (cost < best_cost) { best_cost = cost; best = c; }
  }
  return best;
}

// window for bases that carry all W tables (one shared bucket set): fewer, larger windows pay off.
// Cost in field products: 10 per mixed addition; `bucket_cost` per bucket for everything that scales
// with the bucket count (boundary-partial merge + reduction).  By operation count a bucket costs 38
// (2 full additions + share of the merge), but those kernels run at a lower fraction of the multiplier
// peak than the accumulate kernel: measured on B200 at 2^20 points, c = 20, a bucket costs about as
// much time as 10 mixed additions in G1 and in G2 alike; a sweep of the window over 2^16..2^24 points
// (profiles/r01s2_window_model.md) is matched best by PS_BUCKET_COST = 70 (context.cuh).
inline int msm_pick_window_full(size_t n, double bucket_cost = PS_BUCKET_COST) {
  int best = 4; double best_cost = 1e300;
  for (int c = 4; c <= 24; c++) {
    double W = msm_windows(c);
    if ((double)n * W >= 2.0e9) continue;  // entry indices are 31 bits
    double cost = (double)n * W * 10.0 + (double)(1u << (c - 1)) * bucket_cost;
    if (cost < best_cost) { best_cost = cost; best = c; }
  }
  return best;
}


template <class F> struct PointBytes;
template <> struct PointBytes<Fp> { static constexpr int COMP = 48, AFF = 96; static constexpr int GROUP = PS_G1; };
template <> struct PointBytes<Fp2> { static constexpr int COMP = 96, AFF = 192; static constexpr int GROUP = PS_G2; };

// Every member enqueues kernels on ctx->stream and returns a PS_* status; scratch comes from ctx->arena.
template <class F>
struct GroupOps {
  // the batched Pippenger pipeline (msm.cuh) over base sets that live in one allocation (`slab`; plan.toff gives each
  // output's table offset); results (XYZZ) to d_out[0..plan.nsets)
  static int msm_batch(ps_ctx* ctx, const MsmPlan& plan, const Affine<F>* slab, XYZZ<F>* d_out);
  // wire bytes (device) -> affine Montgomery points; *d_err |= 2 on a bad encoding / a point off the curve,
  // |= 4 on a point outside the prime-order subgroup (checked when subgroup_check is set); d_status (optional) receives
  // those bits per point, 0 for a good one
  static int decode(ps_ctx* ctx, const uint8_t* d_in, size_t n, int format, Affine<F>* d_out, uint32_t* d_err, bool subgroup_check,
                    uint8_t* d_status = nullptr);
  // XYZZ -> affine, one field inversion per few points
  static int to_affine(ps_ctx* ctx, const XYZZ<F>* d_in, size_t n, Affine<F>* d_out);
  // tables t = 1..T-1 of a base set: tab[t][i] = 2^(c t) tab[0][i]
  static int tables_finish(ps_ctx* ctx, Affine<F>* tab, size_t n, int c, int T);
  // out[i] = scalar[i] * generator (standard-form limbs on the device)
  static int from_scalars(ps_ctx* ctx, const uint32_t* d_scalars, size_t n, Affine<F>* d_out);
  static int encode_xyzz(ps_ctx* ctx, const XYZZ<F>* d_pts, size_t count, int format, uint8_t* d_bytes);
  static int encode_affine(ps_ctx* ctx, const Affine<F>* d_pts, size_t count, int format, uint8_t* d_bytes);
  // out[0] = sum of `count` points
  static int sum_points(ps_ctx* ctx, const XYZZ<F>* d_in, uint32_t count, XYZZ<F>* d_out);
  // sums over gathered records (see ps_g16_combine): item i adds, over all `count` records `stride` bytes
  // apart, the points at byte offsets off0[i] and (if >= 0) off1[i]; items <= 2
  static int record_sum(ps_ctx* ctx, int items, uint32_t count, const uint8_t* d_recs, uint32_t stride, const int off0[2],
                        const int off1[2], XYZZ<F>* d_out);
};
extern template struct GroupOps<Fp>;
extern template struct GroupOps<Fp2>;

}  // namespace ps
