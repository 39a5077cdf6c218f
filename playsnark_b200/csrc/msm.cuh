// Pippenger multi-scalar multiplication for G1 and G2 (sm_100a).
//
// Computes what the reference obtains with one scalar multiplication per term:
//   Poly.BlindEval  (algebra.go:348-359)   acc += p[i] * blindedPoint[i]
//   sumBlind        (groth16.go:134-141)   and computeSolCommit (pinochio.go:222-229)
// i.e. the group element  sum_i k_i * P_i ; the affine result is identical whatever the schedule.
//
// Pipeline (all on the device, one stream):
//   1. MsmCountK      signed-digit window decomposition of every scalar (k -> r-k with the point
//                     negated when k > r/2, so small negative witnesses stay short); per-bucket
//                     histogram with the atomic's return value kept as the rank inside the bucket
//   2. exclusive scan bucket offsets
//   3. MsmScatterK    counting-sort of (point index | sign) by bucket
//      (large inputs replace 1-3 with msm_sort_two_level: by partition of buckets, then by bucket per tile)
//   4. MsmAccumK      bucket accumulation: every thread owns L consecutive sorted entries (perfect
//                     balance whatever the scalar distribution), adds the gathered affine bases into
//                     an XYZZ accumulator (madd, 8M+2S), writes buckets that lie wholly inside its
//                     range and emits at most two boundary partials
//   5. MsmRunMergeK / MsmCombineK   merge of the boundary partials (XYZZ + XYZZ): short runs in one
//                     parallel pass, the rest log-depth
//   6. MsmReduceFirstK / MsmReduceK   sum_d d * B_d per bucket set: running sums over small groups, 4-way
//                     weighted merges of (acc, run) pairs, then MsmBitGatherK / MsmPairSumK /
//                     MsmBitFinalK: a low-depth tail by binary decomposition of the weights
//   7. MsmFinalK      Horner over the bucket sets (c*T doublings between sets)
// With T precomputed tables (2^(c t) * P_i, t < T) the windows w = s*T + t share bucket set s.
#pragma once
#include "group_ops.cuh"
#include "team.cuh"

namespace ps {

PS_DEV int msm_seg_of(const MsmPlan& p, uint32_t i) {
  int k = 0;
  while (k + 1 < p.nseg && i >= p.seg[k + 1].start) k++;
  return k;
}

// Where scalar i of the batch comes from and goes to: its scalar array and index in it, the first bucket of its output
// set, the point it multiplies (offset in the slab) and the table stride of that base set.
struct MsmSrc {
  const uint32_t* scalars;
  uint32_t idx, b0, pt, nbase;
  int mont;
};
PS_DEV MsmSrc msm_source(const MsmPlan& p, uint32_t i) {
  MsmSrc s;
  if (p.row_len) {
    const uint32_t set = i / p.row_len;
    s.scalars = p.seg[0].scalars; s.idx = i; s.mont = (int)p.seg[0].mont;
    s.b0 = set * (uint32_t)p.S * p.D; s.nbase = p.nbase[0]; s.pt = p.toff[0] + p.seg[0].first + (i - set * p.row_len);
  } else {
    const MsmSeg sg = p.seg[msm_seg_of(p, i)];
    s.scalars = sg.scalars; s.idx = i - sg.start; s.mont = (int)sg.mont;
    s.b0 = sg.set * (uint32_t)p.S * p.D; s.nbase = p.nbase[sg.set]; s.pt = p.toff[sg.set] + sg.first + s.idx;
  }
  return s;
}

// Loads scalar i (8 LE limbs), optionally leaves Montgomery form, folds k > (r-1)/2 to r-k.
PS_DEV void msm_load_scalar(const uint32_t* scalars, uint32_t i, int mont, uint32_t k[8], bool& neg) {
  Fr x;
#pragma unroll
  for (int j = 0; j < 8; j++) x.v[j] = scalars[(size_t)i * 8 + j];
  if (mont) x = x.from_mont();
  // borrow of HALF - k  <=>  k > HALF
  uint32_t t = ptx_sub_cc(FrParams::HALF(0), x.v[0]);
#pragma unroll
  for (int j = 1; j < 8; j++) t = ptx_subc_cc(FrParams::HALF(j), x.v[j]);
  uint32_t borrow = ptx_subc(0, 0);
  neg = borrow != 0;
  if (neg) {
    uint32_t m[8];
    m[0] = ptx_sub_cc(FrParams::MOD(0), x.v[0]);
#pragma unroll
    for (int j = 1; j < 8; j++) m[j] = ptx_subc_cc(FrParams::MOD(j), x.v[j]);
#pragma unroll
    for (int j = 0; j < 8; j++) x.v[j] = m[j];
  }
#pragma unroll
  for (int j = 0; j < 8; j++) k[j] = x.v[j];
}

// returns the low c bits and shifts the 256-bit value right by c (1 <= c <= 31)
PS_DEV uint32_t msm_take_bits(uint32_t k[8], int c) {
  uint32_t v = k[0] & ((1u << c) - 1);
#pragma unroll
  for (int j = 0; j < 7; j++) k[j] = (k[j] >> c) | (k[j + 1] << (32 - c));
  k[7] >>= c;
  return v;
}

// Signed digit of window w: d in [-2^(c-1)+1, 2^(c-1)]; returns bucket (|d|-1) and sign, or false for 0.
PS_DEV bool msm_next_digit(uint32_t k[8], int c, uint32_t& carry, uint32_t& mag, bool& dneg) {
  uint32_t v = msm_take_bits(k, c) + carry;
  uint32_t half = 1u << (c - 1);
  if (v > half) { mag = (1u << c) - v; dneg = true; carry = 1; }
  else { mag = v; dneg = false; carry = 0; }
  return mag != 0;
}

struct MsmCountK {
  static constexpr int BLOCK = 256;
  PS_DEV static void run(uint32_t i, MsmPlan p, uint32_t* count, uint32_t* ranks) {
    const MsmSrc src = msm_source(p, i);
    uint32_t k[8]; bool neg;
    msm_load_scalar(src.scalars, src.idx, src.mont, k, neg);
    uint32_t carry = 0;
    for (int w = 0; w < p.W; w++) {
      uint32_t mag; bool dneg;
      uint32_t rank = 0xFFFFFFFFu;
      if (msm_next_digit(k, p.c, carry, mag, dneg)) {
        uint32_t b = src.b0 + (uint32_t)(w / p.T) * p.D + (mag - 1);
        rank = ps_atomic_add(count + b, 1u);
      }
      ranks[(size_t)w * p.total + i] = rank;
    }
  }
};

struct MsmScatterK {
  static constexpr int BLOCK = 256;
  PS_DEV static void run(uint32_t i, MsmPlan p, const uint32_t* off, const uint32_t* ranks, uint32_t* ent) {
    const MsmSrc src = msm_source(p, i);
    uint32_t k[8]; bool neg;
    msm_load_scalar(src.scalars, src.idx, src.mont, k, neg);
    uint32_t carry = 0;
    for (int w = 0; w < p.W; w++) {
      uint32_t mag; bool dneg;
      if (msm_next_digit(k, p.c, carry, mag, dneg)) {
        uint32_t b = src.b0 + (uint32_t)(w / p.T) * p.D + (mag - 1);
        uint32_t pos = off[b] + ranks[(size_t)w * p.total + i];
        uint32_t idx = (uint32_t)(w % p.T) * src.nbase + src.pt;
        ent[pos] = idx | ((neg != dneg) ? 0x80000000u : 0u);
      }
    }
  }
};

// last index b in [0, nb) with off[b] <= pos  (off is non-decreasing, off[0] = 0, pos < off[nb])
PS_DEV uint32_t msm_find_bucket(const uint32_t* off, uint32_t nb, uint32_t pos) {
  uint32_t lo = 0, hi = nb;  // invariant: off[lo] <= pos < off[hi]
  while (hi - lo > 1) {
    uint32_t mid = lo + (hi - lo) / 2;
    if (off[mid] <= pos) lo = mid; else hi = mid;
  }
  return lo;
}

template <class F>
PS_DEV Affine<F> msm_load_point(const Affine<F>* tab, uint32_t e) {
  Affine<F> p = tab[e & 0x7FFFFFFFu];
  if (e >> 31) p.y = p.y.neg();
  return p;
}

// slot flags: bit0 = the bucket has partials to the left, bit1 = to the right
#ifndef PS_G1_MINB
#define PS_G1_MINB 3
#endif
#ifndef PS_G2_MINB
#define PS_G2_MINB 2
#endif
#ifndef PS_ACC_BLOCK
#define PS_ACC_BLOCK 128
#endif
template <class F>
struct MsmAccumK {
  static constexpr int BLOCK = PS_ACC_BLOCK;
  // registers: G1 fits 3 resident blocks per SM without spilling; G2 (Fp2) is register-bound
  static constexpr int MIN_BLOCKS = sizeof(F) == sizeof(Fp) ? PS_G1_MINB : PS_G2_MINB;
  using Self = MsmAccumK<F>;
  PS_DEV static void run(uint32_t tid, uint32_t nb, uint32_t L, const Affine<F>* tab, const uint32_t* ent,
                         const uint32_t* off, XYZZ<F>* buckets, XYZZ<F>* slot_pt, int32_t* slot_bid,
                         uint8_t* slot_fl) {
    const uint32_t M = off[nb];
    const uint32_t head = 2 * tid, tail = 2 * tid + 1;
    slot_bid[head] = -1; slot_bid[tail] = -1;
    uint64_t p0 = (uint64_t)tid * L;
    if (p0 >= M) return;
    uint32_t cur = (uint32_t)p0;
    uint32_t end = (M - cur > L) ? cur + L : M;
    uint32_t b = msm_find_bucket(off, nb, cur);
    bool head_open = off[b] < cur;
    uint32_t bend = off[b + 1];
    XYZZ<F> acc = XYZZ<F>::inf();
    // One flat loop of (at most) L iterations: every lane of the warp reaches the madd together; the
    // bucket hand-over is a short predicated block in front of it.
    for (; cur < end; cur++) {
      if (cur == bend) {  // bucket b ended exactly here
        flush(b, acc, head_open, true, head, tail, buckets, slot_pt, slot_bid, slot_fl);
        acc = XYZZ<F>::inf();
        head_open = false;
        b++;
        while (off[b + 1] <= cur) b++;
        bend = off[b + 1];
      }
      // (an L2 prefetch of the next entry's base was measured slightly slower: 79.8 vs 78.8 ms at 2^24 --
      // the other resident warps already cover the gather latency)
      xyzz_madd(acc, msm_load_point(tab, ent[cur]));
    }
    flush(b, acc, head_open, bend <= end, head, tail, buckets, slot_pt, slot_bid, slot_fl);
  }
  PS_DEV static void flush(uint32_t b, const XYZZ<F>& acc, bool head_open, bool closed, uint32_t head, uint32_t tail,
                           XYZZ<F>* buckets, XYZZ<F>* slot_pt, int32_t* slot_bid, uint8_t* slot_fl) {
    if (closed && !head_open) {
      buckets[b] = acc;
    } else {
      uint32_t s = head_open ? head : tail;
      slot_pt[s] = acc;
      slot_bid[s] = (int32_t)b;
      slot_fl[s] = (uint8_t)((head_open ? 1 : 0) | (closed ? 0 : 2));
    }
  }
};

// The tail kernels below are written once against Coop<T>: T = false is one thread per work item (plain
// serial group law), T = true a team of four lanes per work item (team.cuh).  A kernel launched over
// `items` work items needs items * Coop<T>::LANES threads; only the team's first lane stores results.
template <bool T> struct Coop;
template <> struct Coop<false> {
  static constexpr uint32_t LANES = 1;
  PS_DEV explicit Coop(uint32_t&) {}
  template <class F> PS_DEV void add(XYZZ<F>& acc, const XYZZ<F>& q) const { xyzz_add_c(acc, q); }
  template <class F> PS_DEV void dbl(XYZZ<F>& p) const { p = xyzz_dbl_c(p); }
  PS_DEV bool writer() const { return true; }
  PS_DEV bool idle() const { return false; }
  PS_DEV void sync() const {}
};
template <> struct Coop<true> {
  static constexpr uint32_t LANES = TEAM;
  TeamCtx tc;
  PS_DEV explicit Coop(uint32_t& tid) : tc(TeamCtx::of(tid)) { tid >>= 2; }
  template <class F> PS_DEV void add(XYZZ<F>& acc, const XYZZ<F>& q) const { xyzz_add_t(acc, q, tc); }
  template <class F> PS_DEV void dbl(XYZZ<F>& p) const { xyzz_dbl_t(p, tc); }
  PS_DEV bool writer() const { return tc.tl == 0; }
  // host emulation runs the lanes one after the other, each with the plain serial formulas: lanes 1..3
  // would only repeat lane 0's work
  PS_DEV bool idle() const {
#ifdef __CUDA_ARCH__
    return false;
#else
    return tc.tl != 0;
#endif
  }
  PS_DEV void sync() const { tc.sync(); }
};

// Boundary partials of one bucket sit in consecutive chunks: the tail of the chunk where the bucket
// starts, the heads of the chunks it covers entirely, and the head of the chunk where it ends.  The
// work item that owns the starting tail walks that run (up to RUN_MAX chunks), adds it up into the
// bucket and blanks the slots; every run is owned by exactly one item, so the pass is fully
// parallel.  Longer runs (heavily repeated scalars) are left to the log-depth merge below.
template <class F, bool T>
struct MsmRunMergeK {
  static constexpr int BLOCK = 128;
  static constexpr uint32_t RUN_MAX = 32;
  PS_DEV static void run(uint32_t t, uint32_t n_chunks, XYZZ<F>* buckets, XYZZ<F>* slot_pt, int32_t* slot_bid,
                         const uint8_t* slot_fl) {
    Coop<T> co(t);
    if (co.idle()) return;
    const uint32_t a = 2 * t + 1;  // tail of chunk t
    int32_t bid = slot_bid[a];
    if (bid < 0 || slot_fl[a] != 2) return;  // not the start of a run
    uint32_t len = 0;                         // number of following chunks in the run
    for (uint32_t j = 1; j <= RUN_MAX && t + j < n_chunks; j++) {
      uint32_t h = 2 * (t + j);
      if (slot_bid[h] != bid) return;         // malformed / not ours: leave untouched
      if (slot_fl[h] == 1) { len = j; break; }
    }
    if (!len) return;
    XYZZ<F> acc = slot_pt[a];
    for (uint32_t j = 1; j <= len; j++) co.add(acc, slot_pt[2 * (t + j)]);
    co.sync();  // every lane has read the run before it is blanked
    if (!co.writer()) return;
    buckets[bid] = acc;
    slot_bid[a] = -1;
    for (uint32_t j = 1; j <= len; j++) slot_bid[2 * (t + j)] = -1;
  }
};

template <class F, bool T>
struct MsmCombineK {
  static constexpr int BLOCK = 128;
  PS_DEV static void flush(int32_t bid, const XYZZ<F>& acc, bool cl, bool cr, int final_pass, uint32_t tid,
                           XYZZ<F>* buckets, XYZZ<F>* out_pt, int32_t* out_bid, uint8_t* out_fl) {
    if (bid < 0) return;
    if (final_pass || (!cl && !cr)) { buckets[bid] = acc; return; }
    uint32_t s = cl ? 2 * tid : 2 * tid + 1;
    out_pt[s] = acc; out_bid[s] = bid; out_fl[s] = (uint8_t)((cl ? 1 : 0) | (cr ? 2 : 0));
  }
  PS_DEV static void run(uint32_t tid, uint32_t n_in, uint32_t f, const XYZZ<F>* in_pt, const int32_t* in_bid,
                         const uint8_t* in_fl, XYZZ<F>* buckets, XYZZ<F>* out_pt, int32_t* out_bid,
                         uint8_t* out_fl, int final_pass) {
    Coop<T> co(tid);
    if (co.idle()) return;
    const bool wr = co.writer();
    if (wr) { out_bid[2 * tid] = -1; out_bid[2 * tid + 1] = -1; }
    int32_t cur = -1; bool cl = false, cr = false;
    XYZZ<F> acc = XYZZ<F>::inf();
    for (uint32_t i = 0; i < f; i++) {
      uint64_t j = (uint64_t)tid * f + i;
      if (j >= n_in) break;
      int32_t bid = in_bid[j];
      if (bid < 0) continue;
      uint8_t fl = in_fl[j];
      if (bid != cur) {
        if (wr) flush(cur, acc, cl, cr, final_pass, tid, buckets, out_pt, out_bid, out_fl);
        cur = bid; acc = in_pt[j]; cl = fl & 1; cr = (fl & 2) != 0;
      } else {
        co.add(acc, in_pt[j]); cr = (fl & 2) != 0;
      }
    }
    if (wr) flush(cur, acc, cl, cr, final_pass, tid, buckets, out_pt, out_bid, out_fl);
  }
};

// First level of sum_{d=1..D} d * B_d : item (s, j) covers buckets [j*g, (j+1)*g) of set s and
// emits acc = sum_{i<g} (i+1) * B_{jg+i}, run = sum_i B_{jg+i}.
template <class F, bool T>
struct MsmReduceFirstK {
  static constexpr int BLOCK = 128;
  PS_DEV static void run(uint32_t tid, uint32_t D, uint32_t G, uint32_t g, const XYZZ<F>* buckets, XYZZ<F>* acc_out,
                         XYZZ<F>* run_out) {
    Coop<T> co(tid);
    if (co.idle()) return;
    uint32_t s = tid / G, j = tid % G;
    const XYZZ<F>* B = buckets + (size_t)s * D + (size_t)j * g;
    XYZZ<F> rr = XYZZ<F>::inf(), ww = XYZZ<F>::inf();
    for (uint32_t i = g; i-- > 0;) {
      co.add(rr, B[i]);
      co.add(ww, rr);
    }
    if (co.writer()) { acc_out[tid] = ww; run_out[tid] = rr; }
  }
};

// Next levels: item (s, j) merges f consecutive (acc, run) elements, each spanning 2^log_len
// buckets:  acc = sum_i acc_i + 2^log_len * sum_i i * run_i ,  run = sum_i run_i.
template <class F, bool T>
struct MsmReduceK {
  static constexpr int BLOCK = 64;
  PS_DEV static void run(uint32_t tid, uint32_t n_in, uint32_t n_out, uint32_t f, int log_len, const XYZZ<F>* acc_in,
                         const XYZZ<F>* run_in, XYZZ<F>* acc_out, XYZZ<F>* run_out) {
    Coop<T> co(tid);
    if (co.idle()) return;
    uint32_t s = tid / n_out, j = tid % n_out;
    const XYZZ<F>* A = acc_in + (size_t)s * n_in + (size_t)j * f;
    const XYZZ<F>* R = run_in + (size_t)s * n_in + (size_t)j * f;
    XYZZ<F> asum = XYZZ<F>::inf(), rr = XYZZ<F>::inf(), ww = XYZZ<F>::inf();
    for (uint32_t i = f; i-- > 0;) {
      if ((size_t)j * f + i >= n_in) continue;
      co.add(asum, A[i]);
      co.add(rr, R[i]);
      if (i > 0) co.add(ww, rr);
    }
    for (int d = 0; d < log_len; d++) co.dbl(ww);
    co.add(asum, ww);
    if (co.writer()) { acc_out[tid] = asum; run_out[tid] = rr; }
  }
};

// Low-depth tail of the bucket reduction.  With G = 2^g elements (acc_j, run_j) left per set,
//   sum_j acc_j + len * sum_j j * run_j  =  A + len * sum_{k<g} 2^k T_k ,   T_k = sum_{j : bit k of j} run_j ,
// so the tail is g+1 independent plain sums (pairwise trees, one addition deep per launch) and a
// short Horner, instead of a chain of weighted merges with growing doubling counts.
// Y rows per set: row 0 = acc pairs already added, row k+1 = the run_j with bit k of j set; G/2 entries each.
template <class F, bool T>
struct MsmBitGatherK {
  static constexpr int BLOCK = 64;
  PS_DEV static void run(uint32_t tid, uint32_t G, int g, const XYZZ<F>* acc, const XYZZ<F>* run, XYZZ<F>* Y) {
    Coop<T> co(tid);
    if (co.idle()) return;
    const uint32_t half = G / 2;
    uint32_t s = tid / ((uint32_t)(g + 1) * half), rem = tid % ((uint32_t)(g + 1) * half);
    uint32_t r = rem / half, i = rem % half;
    XYZZ<F> y;
    if (r == 0) {
      y = acc[(size_t)s * G + 2 * i];
      co.add(y, acc[(size_t)s * G + 2 * i + 1]);
    } else {
      uint32_t k = r - 1;
      uint32_t j = ((i >> k) << (k + 1)) | (1u << k) | (i & ((1u << k) - 1));
      y = run[(size_t)s * G + j];
    }
    if (co.writer()) Y[tid] = y;
  }
};
// out[row][i] = in[row][2i] + in[row][2i+1];  rows of n_in entries -> rows of n_in/2
template <class F, bool T>
struct MsmPairSumK {
  static constexpr int BLOCK = 64;
  PS_DEV static void run(uint32_t tid, uint32_t n_in, const XYZZ<F>* in, XYZZ<F>* out) {
    Coop<T> co(tid);
    if (co.idle()) return;
    uint32_t half = n_in / 2;
    uint32_t row = tid / half, i = tid % half;
    XYZZ<F> y = in[(size_t)row * n_in + 2 * i];
    co.add(y, in[(size_t)row * n_in + 2 * i + 1]);
    if (co.writer()) out[tid] = y;
  }
};
// per set: R = sum_k 2^k T_k (Horner), out = A + 2^log_len R;  Y holds g+1 single-entry rows per set
template <class F, bool T>
struct MsmBitFinalK {
  static constexpr int BLOCK = 32;
  PS_DEV static void run(uint32_t s, int g, int log_len, const XYZZ<F>* Y, XYZZ<F>* out) {
    Coop<T> co(s);
    if (co.idle()) return;
    const XYZZ<F>* row = Y + (size_t)s * (g + 1);
    XYZZ<F> r = XYZZ<F>::inf();
    for (int k = g - 1; k >= 0; k--) {
      co.dbl(r);
      co.add(r, row[k + 1]);
    }
    for (int d = 0; d < log_len; d++) co.dbl(r);
    co.add(r, row[0]);
    if (co.writer()) out[s] = r;
  }
};

// Horner over the bucket sets of output k: out[k] = sum_s 2^(shift*s) * sets[k*S + s]   (one work item per output)
template <class F, bool T>
struct MsmFinalK {
  static constexpr int BLOCK = 32;
  PS_DEV static void run(uint32_t tid, int S, int shift, const XYZZ<F>* sets, XYZZ<F>* out) {
    Coop<T> co(tid);
    if (co.idle()) return;
    XYZZ<F> r = XYZZ<F>::inf();
    for (int s = S - 1; s >= 0; s--) {
      for (int d = 0; d < shift; d++) co.dbl(r);
      co.add(r, sets[(size_t)tid * S + s]);
    }
    if (co.writer()) out[tid] = r;
  }
};

// sums `count` XYZZ points (multi-GPU partials) into out   (one work item)
template <class F, bool T>
struct MsmSumK {
  static constexpr int BLOCK = 32;
  PS_DEV static void run(uint32_t tid, uint32_t count, const XYZZ<F>* in, XYZZ<F>* out) {
    Coop<T> co(tid);
    if (co.idle()) return;
    if (tid != 0) return;
    XYZZ<F> r = XYZZ<F>::inf();
    for (uint32_t i = 0; i < count; i++) co.add(r, in[i]);
    if (co.writer()) *out = r;
  }
};

// ---- exclusive scan of uint32 counters --------------------------------------------------------------
#if PS_GPU
static constexpr int SCAN_THREADS = 256;
static constexpr int SCAN_ITEMS = 8;
static constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

static __global__ void __launch_bounds__(SCAN_THREADS) k_scan_tiles(const uint32_t* in, uint32_t* out, uint32_t* tile_sums, uint32_t n) {
  __shared__ uint32_t warp_sums[SCAN_THREADS / 32];
  uint32_t base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
  uint32_t v[SCAN_ITEMS];
  uint32_t local = 0;
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; i++) { v[i] = (base + i < n) ? in[base + i] : 0; local += v[i]; }
  uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  uint32_t inc = local;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += t; }
  if (lane == 31) warp_sums[wid] = inc;
  __syncthreads();
  if (wid == 0) {
    uint32_t ws = lane < SCAN_THREADS / 32 ? warp_sums[lane] : 0;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, ws, d); if (lane >= d) ws += t; }
    if (lane < SCAN_THREADS / 32) warp_sums[lane] = ws;
  }
  __syncthreads();
  uint32_t excl = inc - local + (wid ? warp_sums[wid - 1] : 0);
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; i++) { if (base + i < n) out[base + i] = excl; excl += v[i]; }
  if (threadIdx.x == SCAN_THREADS - 1) tile_sums[blockIdx.x] = warp_sums[SCAN_THREADS / 32 - 1];
}
static __global__ void __launch_bounds__(1024) k_scan_sums(uint32_t* sums, uint32_t n) {
  __shared__ uint32_t warp_sums[32];
  __shared__ uint32_t carry_s;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (uint32_t base = 0; base < n; base += 1024) {
    uint32_t idx = base + threadIdx.x;
    uint32_t v = idx < n ? sums[idx] : 0;
    uint32_t inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += t; }
    if (lane == 31) warp_sums[wid] = inc;
    __syncthreads();
    if (wid == 0) {
      uint32_t ws = warp_sums[lane];
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, ws, d); if (lane >= d) ws += t; }
      warp_sums[lane] = ws;
    }
    __syncthreads();
    uint32_t carry = carry_s;
    uint32_t excl = carry + inc - v + (wid ? warp_sums[wid - 1] : 0);
    if (idx < n) sums[idx] = excl;
    __syncthreads();
    if (threadIdx.x == 1023) carry_s = carry + warp_sums[31];
    __syncthreads();
  }
}
static __global__ void __launch_bounds__(SCAN_THREADS) k_scan_add(uint32_t* out, const uint32_t* tile_sums, uint32_t n) {
  uint32_t base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
  uint32_t add = tile_sums[blockIdx.x];
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; i++) if (base + i < n) out[base + i] += add;
}
#endif

// out[i] = sum_{j<i} in[i], i < n (in and out may not alias); tile_sums: scratch of ceil(n/2048)+1
inline int exclusive_scan_u32(ps_stream_t st, const uint32_t* in, uint32_t* out, uint32_t* tile_sums, uint32_t n) {
#if PS_GPU
  uint32_t tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
  k_scan_tiles<<<tiles, SCAN_THREADS, 0, st>>>(in, out, tile_sums, n);
  k_scan_sums<<<1, 1024, 0, st>>>(tile_sums, tiles);
  k_scan_add<<<tiles, SCAN_THREADS, 0, st>>>(out, tile_sums, n);
  PS_CUDA_TRY(cudaGetLastError());
  launch_counter() += 3;
#else
  (void)st; (void)tile_sums;
  uint32_t acc = 0;
  for (uint32_t i = 0; i < n; i++) { uint32_t v = in[i]; out[i] = acc; acc += v; }
#endif
  return PS_OK;
}

// ---- two-level sort for large inputs -------------------------------------------------------------------
// The one-pass counting sort spends one global atomic that returns a value per entry (its rank inside the bucket),
// writes and reads back a rank array as large as the entry array, and scatters single words to random positions
// of an entry array far larger than L2.  Above the automatic threshold the entries are sorted in two levels
// instead.  The bucket b splits into a coarse part, the partition b >> s (about 1024 of them), and a fine part,
// b & (2^s - 1):
//   1. k_sort_part_count: a block of scalars (at most SORT_STAGE entries) builds a shared histogram of its entries'
//      partitions and stores it as one column of a (partition, block) count matrix: no global atomics.
//   2. exclusive scan of that matrix, partition-major: every (block, partition) pair gets its run of the staging
//      arrays, and partition q starts at the run of (block 0, q).
//   3. k_sort_part_scatter: the same blocks decode their scalars once more, rank the entries by partition into a
//      shared-memory stage, and write every run (entry words, and the fine digits, 2 B, beside them) with
//      consecutive threads: runs of ~20 entries at 2^24 points (W = 12), each reaching L2 in one burst.
//   4. k_sort_fine_count: fixed tiles of SORT_TILE staging entries, never straddling a partition, build a shared
//      histogram of their partition's 2^s fine buckets, store it per tile and add it to the bucket counts, one
//      global atomic per (tile, non-empty bucket).
//   5. exclusive scan of the bucket counts into the offsets the accumulation reads.
//   6. k_sort_fine_scatter: the same tiles reload their histogram, reserve a base per (tile, bucket) from a cursor
//      that starts at the bucket's offset, rank their entries by fine bucket into a shared-memory stage and write
//      each bucket's segment to the entry array.  Tiles run in partition order, so the stores land inside the
//      window of the entry array the resident blocks cover (a partition is ~0.8 MB at 2^24 points), in L2.
// Fixed tiles keep the work balanced whatever the scalar distribution: all scalars equal put every entry into
// one partition and one bucket, which then simply has many tiles.  The order inside a bucket is arbitrary, as
// with the atomic ranks of the one-pass sort; the accumulated bucket is the same point.
constexpr int SORT_BLOCK = 1024;                // threads of the block-cooperative sort kernels
constexpr uint32_t SORT_STAGE = 20480;          // entries a coarse block stages in shared memory (8 B each)
constexpr uint32_t SORT_TILE = 16384;           // staging entries per fine tile (6 B each in shared memory)
constexpr int SORT_PARTS_LOG = 10;              // about 2^10 coarse partitions
constexpr int SORT_FINE_LOG_MAX = 13;           // fine histograms: at most 2 x 32 KB of shared memory
constexpr uint32_t SORT_PARTS_MAX = 4096;       // coarse histograms: at most 2 x 16 KB beside the stage

// Calls fn(b, e) for every non-zero digit of scalar i of the batch: b = its bucket, e = its entry word
// (table point | sign), as MsmCountK / MsmScatterK compute them.
template <class Fn>
PS_DEV void msm_for_entries(const MsmPlan& p, uint32_t i, Fn&& fn) {
  const MsmSrc src = msm_source(p, i);
  uint32_t k[8]; bool neg;
  msm_load_scalar(src.scalars, src.idx, src.mont, k, neg);
  uint32_t carry = 0, t = 0, b0 = src.b0, tab = src.pt;
  for (int w = 0; w < p.W; w++) {
    uint32_t mag; bool dneg;
    if (msm_next_digit(k, p.c, carry, mag, dneg)) fn(b0 + (mag - 1), tab | ((neg != dneg) ? 0x80000000u : 0u));
    if (++t == (uint32_t)p.T) { t = 0; b0 += p.D; tab = src.pt; } else { tab += src.nbase; }
  }
}

// fine tile t (t < tile_first[nparts]): its partition q and its range [lo, hi) of the staging arrays
PS_DEV void sort_tile(uint32_t t, uint32_t nparts, const uint32_t* part_off, const uint32_t* tile_first, uint32_t& q,
                      uint32_t& lo, uint32_t& hi) {
  q = msm_find_bucket(tile_first, nparts, t);
  lo = part_off[q] + (t - tile_first[q]) * SORT_TILE;
  hi = part_off[q + 1] - lo > SORT_TILE ? lo + SORT_TILE : part_off[q + 1];
}

// from the scanned (partition, block) matrix: part_off[q] = start of partition q (q <= nparts), and the number of
// fine tiles of each partition, tiles[q] (tiles[nparts] = 0)
struct MsmSortTilesK {
  static constexpr int BLOCK = 256;
  PS_DEV static void run(uint32_t q, uint32_t nparts, uint32_t nblocks, const uint32_t* run_off, uint32_t* part_off,
                         uint32_t* tiles) {
    part_off[q] = run_off[(size_t)q * nblocks];
    tiles[q] = q < nparts ? (run_off[(size_t)(q + 1) * nblocks] - run_off[(size_t)q * nblocks] + SORT_TILE - 1) / SORT_TILE : 0;
  }
};

#if PS_GPU
// ctr[key]++ in shared memory for the calling lanes; returns the old value.  When all active lanes of the warp hit
// the same counter (skewed scalars), one atomic serves them all.
static __device__ __forceinline__ uint32_t sort_sh_inc(uint32_t* ctr, uint32_t key) {
  const uint32_t act = __activemask();
  const int lead = __ffs(act) - 1;
  if (__all_sync(act, key == __shfl_sync(act, key, lead))) {
    const uint32_t lane = threadIdx.x & 31;
    uint32_t base = 0;
    if ((int)lane == lead) base = atomicAdd(&ctr[key], (uint32_t)__popc(act));
    return __shfl_sync(act, base, lead) + __popc(act & ((1u << lane) - 1));
  }
  return atomicAdd(&ctr[key], 1u);
}

// In-place exclusive scan of the n shared counters c[0..n) by the whole block; c[n] receives the total.
static __device__ void sort_block_scan(uint32_t* c, uint32_t n) {
  __shared__ uint32_t warp_tot[SORT_BLOCK / 32];
  const uint32_t per = (n + SORT_BLOCK - 1) / SORT_BLOCK, a = threadIdx.x * per, e = a + per < n ? a + per : n;
  uint32_t local = 0;
  for (uint32_t k = a; k < e; k++) local += c[k];
  const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  uint32_t inc = local;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += t; }
  if (lane == 31) warp_tot[wid] = inc;
  __syncthreads();
  if (wid == 0) {
    uint32_t ws = warp_tot[lane];
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, ws, d); if (lane >= d) ws += t; }
    warp_tot[lane] = ws;
  }
  __syncthreads();
  uint32_t run = inc - local + (wid ? warp_tot[wid - 1] : 0);
  for (uint32_t k = a; k < e; k++) { const uint32_t v = c[k]; c[k] = run; run += v; }
  if (threadIdx.x == SORT_BLOCK - 1) c[n] = run;
  __syncthreads();
}

static __global__ void __launch_bounds__(SORT_BLOCK) k_sort_part_count(MsmPlan p, uint32_t spb, int s, uint32_t nparts,
                                                                     uint32_t* run_count) {
  extern __shared__ uint32_t sh_sort[];
  for (uint32_t q = threadIdx.x; q < nparts; q += SORT_BLOCK) sh_sort[q] = 0;
  __syncthreads();
  const uint32_t i0 = blockIdx.x * spb, i1 = p.total - i0 > spb ? i0 + spb : p.total;
  for (uint32_t i = i0 + threadIdx.x; i < i1; i += SORT_BLOCK)
    msm_for_entries(p, i, [&](uint32_t b, uint32_t) { sort_sh_inc(sh_sort, b >> s); });
  __syncthreads();
  for (uint32_t q = threadIdx.x; q < nparts; q += SORT_BLOCK) run_count[(size_t)q * gridDim.x + blockIdx.x] = sh_sort[q];
}

// Both scatters write through shared memory: a block ranks its entries by key (partition, or fine bucket) into a
// stage ordered by key, with the key beside each entry, and then writes the stage with consecutive threads, so
// every run reaches L2 in one burst of whole sectors instead of word by word over the block's lifetime.
// Shared layout: cnt[nk + 1] (counts, then cursors, then run base - stage offset), loc[nk + 1] (the stage's key
// offsets), then the stage.
static __global__ void __launch_bounds__(SORT_BLOCK) k_sort_part_scatter(MsmPlan p, uint32_t spb, int s, uint32_t nparts,
                                                                       const uint32_t* run_off, uint32_t* st_ent,
                                                                       uint16_t* st_fine) {
  extern __shared__ uint32_t sh_sort[];
  uint32_t* cnt = sh_sort;
  uint32_t* loc = cnt + nparts + 1;
  uint32_t* s_ent = loc + nparts + 1;
  uint16_t* s_fine = reinterpret_cast<uint16_t*>(s_ent + SORT_STAGE);
  uint16_t* s_part = s_fine + SORT_STAGE;
  const uint32_t nblocks = gridDim.x;
  for (uint32_t q = threadIdx.x; q < nparts; q += SORT_BLOCK) {
    const size_t r = (size_t)q * nblocks + blockIdx.x;
    cnt[q] = run_off[r + 1] - run_off[r];
  }
  __syncthreads();
  sort_block_scan(cnt, nparts);
  for (uint32_t q = threadIdx.x; q <= nparts; q += SORT_BLOCK) loc[q] = cnt[q];
  __syncthreads();
  const uint32_t i0 = blockIdx.x * spb, i1 = p.total - i0 > spb ? i0 + spb : p.total;
  const uint32_t fmask = (1u << s) - 1;
  for (uint32_t i = i0 + threadIdx.x; i < i1; i += SORT_BLOCK)
    msm_for_entries(p, i, [&](uint32_t b, uint32_t e) {
      const uint32_t j = sort_sh_inc(cnt, b >> s);
      s_ent[j] = e;
      s_fine[j] = (uint16_t)(b & fmask);
      s_part[j] = (uint16_t)(b >> s);
    });
  __syncthreads();
  for (uint32_t q = threadIdx.x; q < nparts; q += SORT_BLOCK) cnt[q] = run_off[(size_t)q * nblocks + blockIdx.x] - loc[q];
  __syncthreads();
  const uint32_t m = loc[nparts];
  for (uint32_t j = threadIdx.x; j < m; j += SORT_BLOCK) {
    const uint32_t pos = cnt[s_part[j]] + j;
    st_ent[pos] = s_ent[j];
    st_fine[pos] = s_fine[j];
  }
}

static __global__ void __launch_bounds__(SORT_BLOCK) k_sort_fine_count(int s, uint32_t nparts, const uint32_t* part_off,
                                                                     const uint32_t* tile_first, const uint16_t* st_fine,
                                                                     uint32_t* tile_count, uint32_t* count) {
  extern __shared__ uint32_t sh_sort[];
  if (blockIdx.x >= tile_first[nparts]) return;
  uint32_t q, lo, hi;
  sort_tile(blockIdx.x, nparts, part_off, tile_first, q, lo, hi);
  for (uint32_t f = threadIdx.x; f < (1u << s); f += SORT_BLOCK) sh_sort[f] = 0;
  __syncthreads();
  for (uint32_t j = lo + threadIdx.x; j < hi; j += SORT_BLOCK) sort_sh_inc(sh_sort, st_fine[j]);
  __syncthreads();
  for (uint32_t f = threadIdx.x; f < (1u << s); f += SORT_BLOCK) {
    const uint32_t n = sh_sort[f];
    tile_count[((size_t)blockIdx.x << s) + f] = n;
    if (n) atomicAdd(&count[(q << s) + f], n);
  }
}

static __global__ void __launch_bounds__(SORT_BLOCK) k_sort_fine_scatter(int s, uint32_t nparts, const uint32_t* part_off,
                                                                       const uint32_t* tile_first, const uint32_t* tile_count,
                                                                       const uint16_t* st_fine, const uint32_t* st_ent,
                                                                       uint32_t* cur, uint32_t* ent) {
  extern __shared__ uint32_t sh_sort[];
  if (blockIdx.x >= tile_first[nparts]) return;
  const uint32_t nf = 1u << s;
  uint32_t* cnt = sh_sort;
  uint32_t* loc = cnt + nf + 1;
  uint32_t* s_ent = loc + nf + 1;
  uint16_t* s_fine = reinterpret_cast<uint16_t*>(s_ent + SORT_TILE);
  uint32_t q, lo, hi;
  sort_tile(blockIdx.x, nparts, part_off, tile_first, q, lo, hi);
  for (uint32_t f = threadIdx.x; f < nf; f += SORT_BLOCK) cnt[f] = tile_count[((size_t)blockIdx.x << s) + f];
  __syncthreads();
  sort_block_scan(cnt, nf);
  for (uint32_t f = threadIdx.x; f <= nf; f += SORT_BLOCK) loc[f] = cnt[f];
  __syncthreads();
  for (uint32_t j = lo + threadIdx.x; j < hi; j += SORT_BLOCK) {
    const uint32_t f = st_fine[j], k = sort_sh_inc(cnt, f);
    s_ent[k] = st_ent[j];
    s_fine[k] = (uint16_t)f;
  }
  __syncthreads();
  for (uint32_t f = threadIdx.x; f < nf; f += SORT_BLOCK) {
    const uint32_t n = loc[f + 1] - loc[f];
    if (n) cnt[f] = atomicAdd(&cur[(q << s) + f], n) - loc[f];
  }
  __syncthreads();
  for (uint32_t j = threadIdx.x; j < hi - lo; j += SORT_BLOCK) ent[cnt[s_fine[j]] + j] = s_ent[j];
}
#endif

// Two-level sort of the batch's entries by bucket (s, nparts as chosen by msm_run_batch): leaves the bucket offsets
// in off[0..nb] and the entries in ent.  count (nb + 1 words) must be zero.  Host emulation: the block-cooperative
// kernels become serial loops (one block, one tile at a time) that produce the same offsets and a valid order.
inline int msm_sort_two_level(ps_stream_t st, Arena& ar, const MsmPlan& g, uint32_t nb, int s, uint32_t nparts, uint32_t* count,
                              uint32_t* off, uint32_t* tile_sums, uint32_t* ent) {
  const size_t max_ent = (size_t)g.total * g.W;
  const uint32_t spb = SORT_STAGE / (uint32_t)g.W;  // scalars per coarse block: its entries fit the stage
  const uint32_t nblocks = (g.total + spb - 1) / spb;
  const size_t runs = (size_t)nparts * nblocks;     // (partition, block) pairs
  const size_t max_tiles = (max_ent + SORT_TILE - 1) / SORT_TILE + nparts;
  uint32_t* run_count = ar.take<uint32_t>(runs + 1);
  uint32_t* run_off = ar.take<uint32_t>(runs + 1);
  uint32_t* run_sums = ar.take<uint32_t>(runs / 2048 + 2);
  uint32_t* part_off = ar.take<uint32_t>(nparts + 1);
  uint32_t* tiles = ar.take<uint32_t>(nparts + 1);
  uint32_t* tile_first = ar.take<uint32_t>(nparts + 1);
  uint32_t* tile_count = ar.take<uint32_t>(max_tiles << s);
  uint32_t* st_ent = ar.take<uint32_t>(max_ent);
  uint16_t* st_fine = ar.take<uint16_t>(max_ent);
  if (!run_count || !run_off || !run_sums || !part_off || !tiles || !tile_first || !tile_count || !st_ent || !st_fine)
    return PS_ERR_ALLOC;
  PS_TRY(dev_memset(run_count + runs, 0, 4, st));
#if PS_GPU
  const size_t part_smem = (2 * (size_t)nparts + 2) * 4 + (size_t)SORT_STAGE * 8;
  const size_t fine_smem = (2 * ((size_t)1 << s) + 2) * 4 + (size_t)SORT_TILE * 6;
  PS_CUDA_TRY(cudaFuncSetAttribute(k_sort_part_scatter, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)part_smem));
  PS_CUDA_TRY(cudaFuncSetAttribute(k_sort_fine_scatter, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fine_smem));
  k_sort_part_count<<<nblocks, SORT_BLOCK, nparts * 4, st>>>(g, spb, s, nparts, run_count);
  PS_CUDA_TRY(cudaGetLastError());
  launch_counter()++;
#else
  PS_TRY(dev_memset(run_count, 0, runs * 4, st));
  for (uint32_t i = 0; i < g.total; i++)
    msm_for_entries(g, i, [&](uint32_t b, uint32_t) { run_count[(size_t)(b >> s) * nblocks + i / spb]++; });
#endif
  PS_TRY(exclusive_scan_u32(st, run_count, run_off, run_sums, (uint32_t)runs + 1));
  PS_LAUNCH(MsmSortTilesK, st, (size_t)nparts + 1, nparts, nblocks, (const uint32_t*)run_off, part_off, tiles);
  PS_TRY(exclusive_scan_u32(st, tiles, tile_first, tile_sums, nparts + 1));
#if PS_GPU
  k_sort_part_scatter<<<nblocks, SORT_BLOCK, part_smem, st>>>(g, spb, s, nparts, run_off, st_ent, st_fine);
  PS_CUDA_TRY(cudaGetLastError());
  launch_counter()++;
  k_sort_fine_count<<<(uint32_t)max_tiles, SORT_BLOCK, 4u << s, st>>>(s, nparts, part_off, tile_first, st_fine, tile_count, count);
  PS_CUDA_TRY(cudaGetLastError());
  launch_counter()++;
#else
  for (uint32_t i = 0; i < g.total; i++)  // run_count[r] counts down the entries run r still has to take
    msm_for_entries(g, i, [&](uint32_t b, uint32_t e) {
      const size_t r = (size_t)(b >> s) * nblocks + i / spb;
      const uint32_t pos = run_off[r + 1] - run_count[r]--;
      st_ent[pos] = e;
      st_fine[pos] = (uint16_t)(b & ((1u << s) - 1));
    });
  for (uint32_t t = 0; t < tile_first[nparts]; t++) {
    uint32_t q, lo, hi;
    sort_tile(t, nparts, part_off, tile_first, q, lo, hi);
    for (uint32_t j = lo; j < hi; j++) count[(q << s) + st_fine[j]]++;
  }
#endif
  PS_TRY(exclusive_scan_u32(st, count, off, tile_sums, nb + 1));
  PS_TRY(dev_d2d(count, off, (size_t)nb * 4, st));  // from here on: the buckets' cursors
#if PS_GPU
  k_sort_fine_scatter<<<(uint32_t)max_tiles, SORT_BLOCK, fine_smem, st>>>(s, nparts, part_off, tile_first, tile_count, st_fine,
                                                                         st_ent, count, ent);
  PS_CUDA_TRY(cudaGetLastError());
  launch_counter()++;
#else
  for (uint32_t t = 0; t < tile_first[nparts]; t++) {
    uint32_t q, lo, hi;
    sort_tile(t, nparts, part_off, tile_first, q, lo, hi);
    for (uint32_t j = lo; j < hi; j++) ent[count[(q << s) + st_fine[j]]++] = st_ent[j];
  }
#endif
  return PS_OK;
}

// the hot kernel: G1 as is; G2 through the layout-identical Fp2I (inlined base-field products)
template <class F>
inline int launch_accum(ps_stream_t st, size_t T1, uint32_t nb, uint32_t L, const Affine<F>* tab, const uint32_t* ent, const uint32_t* off,
                        XYZZ<F>* buckets, XYZZ<F>* slot_pt, int32_t* slot_bid, uint8_t* slot_fl) {
  PS_LAUNCH(MsmAccumK<F>, st, T1, nb, L, tab, ent, off, buckets, slot_pt, slot_bid, slot_fl);
  return PS_OK;
}
// defined in accum_g2.cu (its own translation unit: the fully inlined kernel dominates compile time)
int launch_accum_g2(ps_stream_t st, size_t T1, uint32_t nb, uint32_t L, const Affine<Fp2>* tab, const uint32_t* ent, const uint32_t* off,
                    XYZZ<Fp2>* buckets, XYZZ<Fp2>* slot_pt, int32_t* slot_bid, uint8_t* slot_fl);
template <>
inline int launch_accum<Fp2>(ps_stream_t st, size_t T1, uint32_t nb, uint32_t L, const Affine<Fp2>* tab, const uint32_t* ent,
                             const uint32_t* off, XYZZ<Fp2>* buckets, XYZZ<Fp2>* slot_pt, int32_t* slot_bid, uint8_t* slot_fl) {
  return launch_accum_g2(st, T1, nb, L, tab, ent, off, buckets, slot_pt, slot_bid, slot_fl);
}

// Launches tail kernel K over `items` work items: a team of four lanes per item when the grid is small
// enough to be latency-bound (a few waves), one thread per item when it is throughput-bound.
#ifndef PS_TEAM_MAX_ITEMS
#define PS_TEAM_MAX_ITEMS 65536
#endif
template <template <class, bool> class K, class F, class... Args>
inline int launch_coop(bool team, ps_stream_t st, size_t items, Args... args) {
  if (team && items <= PS_TEAM_MAX_ITEMS) return ps_launch<K<F, true>>(st, items * TEAM, args...);
  return ps_launch<K<F, false>>(st, items, args...);
}

// Runs the pipeline for a batch (plan + per-output tables); the nsets results (XYZZ) go to d_out[0..nsets).
template <class F>
int msm_run_batch(ps_ctx* ctx, const MsmPlan& g, const Affine<F>* tab, XYZZ<F>* d_out) {
  ps_stream_t st = ctx->stream;
  Arena& ar = ctx->arena;
  if (g.nsets < 1 || (g.nsets > MSM_MAX_SEG && !g.row_len) || g.nseg < 0 || g.nseg > MSM_MAX_SEG) return PS_ERR_ARG;
  if (g.row_len && (g.nseg != 1 || (uint64_t)g.nsets * g.row_len != g.total)) return PS_ERR_ARG;
  if (g.total == 0) return dev_memset(d_out, 0, (size_t)g.nsets * sizeof(XYZZ<F>), st);
  const int S_all = g.nsets * g.S;                 // bucket sets of the whole batch
  const uint32_t nb = (uint32_t)S_all * g.D;
  const size_t max_ent = (size_t)g.total * g.W;
  if (max_ent >= 0xFFFFFFFFull || (uint64_t)S_all * g.D >= 0x7FFFFFFFull) return PS_ERR_UNSUPPORTED;

  // entries per accumulate thread.  Target L0: about one average bucket or more, so that a bucket spans
  // at most two or three threads (few boundary partials, short merge runs); twice that when the input
  // is large enough to keep > 400K threads.  Then whole WAVES: the kernel keeps R = SMs x blocks/SM x 128
  // threads resident and every thread runs the same L iterations, so a grid of 1.1 R threads costs as
  // much as one of 2 R (measured: 2^20 points at c = 17 took 9.3 ms in 61K threads of 256 entries,
  // 1.08 waves).  w = number of waves at about L0 entries per thread; L is then set so that the grid
  // fills exactly w waves.
  const size_t avg_bucket = max_ent / nb + 1;
  uint32_t L0 = 8;
  while (L0 < 512 && L0 < avg_bucket) L0 <<= 1;
  if (L0 < 512 && max_ent / (2 * (size_t)L0) >= 400000) L0 <<= 1;
  const size_t R = (size_t)ctx->sm_count * MsmAccumK<F>::MIN_BLOCKS * MsmAccumK<F>::BLOCK;
  // With SHORT chunks (L0 <= 128: small MSMs, few entries per bucket) the wave count is rounded DOWN instead (option
  // msm_wave_floor, default): chunks of L0 .. 2 L0 entries instead of L0/2 .. L0, i.e. the same accumulation work in
  // half as many chunks -- half the boundary partials, slot writes and merge items, which is what the shard-sized MSMs
  // of the multi-GPU prover spend a third of their time on (G1, 2^17 points: 2.34 -> 1.91 ms; 8-GPU proof 12.5 -> 11.6 ms).
  // Long chunks amortise that overhead anyway and prefer the better balance of two waves (G2, 2^20 points, L0 = 256:
  // one wave of 415 entries was 0.35 ms slower than two of 207).
  size_t waves = (max_ent + R * L0 - 1) / (R * L0);
  if (ctx->msm_wave_floor && L0 <= 128 && waves > 1 && waves < 6) waves = max_ent / (R * L0);
  // with many waves the last, partly filled one costs little and L0 itself is kept (more, shorter chunks
  // only add boundary partials: measured +0.2 ms of merge at 2^20, c = 20, for no gain in the accumulation)
  uint32_t L = waves >= 6 ? L0 : (uint32_t)((max_ent + waves * R - 1) / (waves * R));
  if (L < 8) L = 8;
  const size_t T1 = (max_ent + L - 1) / L;
  const uint32_t CF = 64;  // slots merged per combine thread (most are empty after the pair merge)
  const bool team = ctx->msm_team != 0;

  uint32_t* count = ar.take<uint32_t>((size_t)nb + 1);
  uint32_t* off = ar.take<uint32_t>((size_t)nb + 1);
  uint32_t* tile_sums = ar.take<uint32_t>((size_t)nb / 2048 + 2);
  uint32_t* ent = ar.take<uint32_t>(max_ent);
  XYZZ<F>* buckets = ar.take<XYZZ<F>>(nb);
  if (!count || !off || !tile_sums || !ent || !buckets) return PS_ERR_ALLOC;

  // sort: the one-pass counting sort for small inputs, the two-level sort from 2^25 entries (measured on B200: one
  // pass is 0.04 ms faster at 2^20 points, 1.6e7 entries; two levels 0.21 ms faster at 2^22 points, 5.5e7 entries).
  // Option msm_scatter: 0 = always one pass, 1 = automatic, 2 = two levels whenever the partition histogram fits.
  int s = 0;
  while (s < SORT_FINE_LOG_MAX && (((uint64_t)nb + (1u << s) - 1) >> s) > (1u << SORT_PARTS_LOG)) s++;
  const uint32_t nparts = (uint32_t)(((uint64_t)nb + (1u << s) - 1) >> s);
  const bool two_level = nparts <= SORT_PARTS_MAX &&
                         (ctx->msm_scatter == 2 || (ctx->msm_scatter == 1 && max_ent >= ((size_t)1 << 25)));

  ctx->ev_valid = false;
  PS_TRY(ctx_event(ctx, 0));
  PS_TRY(dev_memset(count, 0, ((size_t)nb + 1) * 4, st));
  PS_TRY(dev_memset(buckets, 0, (size_t)nb * sizeof(XYZZ<F>), st));
  if (two_level) {
    PS_TRY(msm_sort_two_level(st, ar, g, nb, s, nparts, count, off, tile_sums, ent));
  } else {
    uint32_t* ranks = ar.take<uint32_t>(max_ent);
    if (!ranks) return PS_ERR_ALLOC;
    PS_LAUNCH(MsmCountK, st, g.total, g, count, ranks);
    PS_TRY(exclusive_scan_u32(st, count, off, tile_sums, nb + 1));
    PS_LAUNCH(MsmScatterK, st, g.total, g, (const uint32_t*)off, (const uint32_t*)ranks, ent);
  }
  PS_TRY(ctx_event(ctx, 1));
  {
    size_t slots_a = 2 * T1, slots_b = 2 * ((slots_a + CF - 1) / CF);
    XYZZ<F>* sp[2] = {ar.take<XYZZ<F>>(slots_a), ar.take<XYZZ<F>>(slots_b)};
    int32_t* sb[2] = {ar.take<int32_t>(slots_a), ar.take<int32_t>(slots_b)};
    uint8_t* sf[2] = {ar.take<uint8_t>(slots_a), ar.take<uint8_t>(slots_b)};
    if (!sp[0] || !sp[1] || !sb[0] || !sb[1] || !sf[0] || !sf[1]) return PS_ERR_ALLOC;
    PS_TRY((launch_accum<F>(st, T1, nb, L, tab, ent, off, buckets, sp[0], sb[0], sf[0])));
    PS_TRY(ctx_event(ctx, 2));
    PS_TRY((launch_coop<MsmRunMergeK, F>(team, st, T1, (uint32_t)T1, buckets, sp[0], sb[0], (const uint8_t*)sf[0])));
    {
      size_t n_in = slots_a;
      int cur = 0;
      for (;;) {
        size_t threads = (n_in + CF - 1) / CF;
        int final_pass = threads == 1;
        PS_TRY((launch_coop<MsmCombineK, F>(team, st, threads, (uint32_t)n_in, CF, (const XYZZ<F>*)sp[cur], (const int32_t*)sb[cur],
                                            (const uint8_t*)sf[cur], buckets, sp[cur ^ 1], sb[cur ^ 1], sf[cur ^ 1], final_pass)));
        if (final_pass) break;
        n_in = 2 * threads;
        cur ^= 1;
      }
    }
  }
  PS_TRY(ctx_event(ctx, 3));
  // bucket reduction
  {
    // first level: group size a power of two, about 128K threads
    uint32_t gsz = 1;
    while ((uint64_t)S_all * (g.D / gsz) > 131072 && gsz < g.D) gsz <<= 1;
    if (gsz < 2 && g.D >= 2) gsz = 2;
    if (gsz > g.D) gsz = g.D;
    uint32_t G = g.D / gsz;
    size_t e0 = (size_t)S_all * G;
    XYZZ<F>* accv[2] = {ar.take<XYZZ<F>>(e0), ar.take<XYZZ<F>>(e0 / 2 + S_all)};
    XYZZ<F>* runv[2] = {ar.take<XYZZ<F>>(e0), ar.take<XYZZ<F>>(e0 / 2 + S_all)};
    if (!accv[0] || !accv[1] || !runv[0] || !runv[1]) return PS_ERR_ALLOC;
    PS_TRY((launch_coop<MsmReduceFirstK, F>(team && e0 <= 32768, st, e0, g.D, G, gsz, (const XYZZ<F>*)buckets, accv[0], runv[0])));
    uint32_t n_in = G;
    int log_len = 0;
    while ((1u << log_len) < gsz) log_len++;
    int cur = 0;
    // a few 4-way weighted merges while plenty of elements remain (work-bound levels)
    while (n_in > 8192) {
      uint32_t f = 4, n_out = n_in / f;
      PS_TRY((launch_coop<MsmReduceK, F>(team, st, (size_t)S_all * n_out, n_in, n_out, f, log_len, (const XYZZ<F>*)accv[cur],
                                         (const XYZZ<F>*)runv[cur], accv[cur ^ 1], runv[cur ^ 1])));
      log_len += 2;
      n_in = n_out;
      cur ^= 1;
    }
    XYZZ<F>* sets = accv[cur];
    if (n_in > 1) {
      // low-depth tail: g+1 plain pairwise sums per set, then a short Horner
      int gb = 0;
      while ((1u << gb) < n_in) gb++;
      const uint32_t half = n_in / 2;
      size_t rows = (size_t)S_all * (gb + 1);
      XYZZ<F>* Y[2] = {ar.take<XYZZ<F>>(rows * half), ar.take<XYZZ<F>>(rows * (half / 2 + 1))};
      XYZZ<F>* set_out = ar.take<XYZZ<F>>(S_all);
      if (!Y[0] || !Y[1] || !set_out) return PS_ERR_ALLOC;
      PS_TRY((launch_coop<MsmBitGatherK, F>(team, st, rows * half, n_in, gb, (const XYZZ<F>*)accv[cur], (const XYZZ<F>*)runv[cur], Y[0])));
      int yc = 0;
      for (uint32_t w = half; w > 1; w >>= 1) {
        PS_TRY((launch_coop<MsmPairSumK, F>(team, st, rows * (w / 2), w, (const XYZZ<F>*)Y[yc], Y[yc ^ 1])));
        yc ^= 1;
      }
      PS_TRY((launch_coop<MsmBitFinalK, F>(team, st, (size_t)S_all, gb, log_len, (const XYZZ<F>*)Y[yc], set_out)));
      sets = set_out;
    }
    PS_TRY((launch_coop<MsmFinalK, F>(team, st, (size_t)g.nsets, g.S, g.c * g.T, (const XYZZ<F>*)sets, d_out)));
  }
  PS_TRY(ctx_event(ctx, 4));
  ctx->ev_valid = true;
  return PS_OK;
}

}  // namespace ps
