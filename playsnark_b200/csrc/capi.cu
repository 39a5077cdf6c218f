// C ABI of libplaysnark_b200.so, part 1 (see include/playsnark_b200.h for the contract and the reference
// interfaces each entry point stands in for): contexts, resident base sets, the MSM entry points, key
// loaders and the assembly of Groth16 / PHGR13 proofs.  Host orchestration only: the group kernels are
// reached through GroupOps<F> (group_ops.cuh; instantiated in group_g1.cu / group_g2.cu), the Fr
// polynomial side through poly_api.cuh (capi_poly.cu).
#include <cstdlib>
#include "group_ops.cuh"
#include "microbench.cuh"
#include "multi_api.cuh"

#include <algorithm>
#include <new>

using namespace ps;

namespace {

inline size_t point_bytes(int group, int format) {
  return group == PS_G1 ? (format == PS_FMT_COMPRESSED ? 48 : 96) : (format == PS_FMT_COMPRESSED ? 96 : 192);
}

// Joins the secondary stream back into the primary one on every exit path after a fork, so that an early
// error return cannot leave stream2 work in flight on scratch the next call recycles.
struct ForkGuard {
  ps_ctx* ctx;
  bool joined = false;
  explicit ForkGuard(ps_ctx* c) : ctx(c) {}
  int join() { joined = true; return ctx_join(ctx); }
  ~ForkGuard() {
    if (!joined) { ctx_join(ctx); dev_sync(ctx->stream); }
  }
};

// `shards`: the base set will be summed in `shards` index ranges (one per GPU of a sharded proof); the
// automatic window is sized for n / shards points per call so that each rank's bucket set (whose
// merge and reduction are a fixed cost per call) matches its share
int bases_alloc(int group, size_t n, int window_bits, int tables, int shards, int bucket_cost, ps_bases** out) {
  if (window_bits < 0 || window_bits > 24 || (window_bits > 0 && window_bits < 2)) return PS_ERR_ARG;
  if (tables < 0) {  // automatic: all windows precomputed when the tables fit comfortably in HBM
    if (window_bits == 0) window_bits = msm_pick_window_full(n / (size_t)(shards > 0 ? shards : 1) + 1, (double)bucket_cost);
    tables = msm_windows(window_bits);
    size_t need = n * (size_t)tables * (group == PS_G1 ? sizeof(G1Affine) : sizeof(G2Affine));
    size_t free_b = need * 8, total_b = 0;
#if PS_GPU
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) free_b = 0;
#endif
    (void)total_b;
    if (need > free_b / 4) { tables = 1; window_bits = 0; }
  }
  if (tables < 1) tables = 1;
  if (tables > 1 && window_bits == 0) return PS_ERR_ARG;
  if (window_bits && tables > msm_windows(window_bits)) tables = msm_windows(window_bits);
  if ((unsigned long long)n * (unsigned long long)tables >= 0x7FFFFFFFull) return PS_ERR_UNSUPPORTED;
  ps_bases* b = new (std::nothrow) ps_bases();
  if (!b) return PS_ERR_ALLOC;
  b->group = group; b->n = n; b->c = window_bits; b->T = tables;
  size_t pt = group == PS_G1 ? sizeof(G1Affine) : sizeof(G2Affine);
  int rc = dev_alloc(&b->tab, n * tables * pt);
  if (rc != PS_OK) { delete b; return rc; }
  b->slab = b->tab;
  *out = b;
  return PS_OK;
}

// `nsets` base sets of one group, all with window `window_bits` and all its tables, carved out of ONE device allocation
// (*slab_out, owned by the caller) so that their MSMs can run as one batched pipeline
int bases_alloc_slab(int group, const size_t* counts, int nsets, int window_bits, void** slab_out, ps_bases** out) {
  if (window_bits < 2 || window_bits > 24) return PS_ERR_ARG;
  const size_t pt = group == PS_G1 ? sizeof(G1Affine) : sizeof(G2Affine);
  int tables = msm_windows(window_bits);
  size_t total = 0;
  for (int i = 0; i < nsets; i++) total += counts[i];
  size_t free_b = total * tables * pt * 8, total_b = 0;
#if PS_GPU
  if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) free_b = 0;
#endif
  (void)total_b;
  if (total * tables * pt > free_b / 4) tables = 1;   // not enough HBM for all windows: one table, per-window bucket sets
  if ((unsigned long long)total * (unsigned long long)tables >= 0x7FFFFFFFull) return PS_ERR_UNSUPPORTED;
  void* slab = nullptr;
  PS_TRY(dev_alloc(&slab, total * tables * pt));
  size_t off = 0;
  for (int i = 0; i < nsets; i++) {
    ps_bases* b = new (std::nothrow) ps_bases();
    if (!b) { for (int j = 0; j < i; j++) { delete out[j]; out[j] = nullptr; } dev_free(slab); return PS_ERR_ALLOC; }
    b->group = group; b->n = counts[i]; b->c = window_bits; b->T = tables;
    b->tab = (char*)slab + off * pt; b->slab = slab; b->owns = false;
    off += counts[i] * tables;
    out[i] = b;
  }
  *slab_out = slab;
  return PS_OK;
}

// decodes `b->n` host points into the first table of an allocated base set and builds the other tables
template <class F>
int bases_fill_t(ps_ctx* ctx, ps_bases* b, const uint8_t* points, int format) {
  ps_stream_t st = ctx->stream;
  const size_t n = b->n, bytes = n * point_bytes(PointBytes<F>::GROUP, format);
  uint8_t* d_in = ctx->arena.take<uint8_t>(bytes);
  uint32_t* d_err = ctx->arena.take<uint32_t>(1);
  if (!d_in || !d_err) return PS_ERR_ALLOC;
  if (bytes) PS_TRY(dev_h2d(d_in, points, bytes, st));
  PS_TRY(dev_memset(d_err, 0, 4, st));
  PS_TRY(GroupOps<F>::decode(ctx, d_in, n, format, (Affine<F>*)b->tab, d_err, ctx->subgroup_check != 0));
  PS_TRY(GroupOps<F>::tables_finish(ctx, (Affine<F>*)b->tab, b->n, b->c, b->T));
  uint32_t herr = 0;
  PS_TRY(dev_d2h(&herr, d_err, 4, st));
  PS_TRY(dev_sync(st));
  return herr ? PS_ERR_ENCODING : PS_OK;
}

template <class F>
int bases_load_t(ps_ctx* ctx, const uint8_t* points, size_t n, int format, int window_bits, int tables, ps_bases** out) {
  ps_bases* b = nullptr;
  PS_TRY(bases_alloc(PointBytes<F>::GROUP, n, window_bits, tables, ctx->msm_shards, ctx->msm_bucket_cost, &b));
  int rc = bases_fill_t<F>(ctx, b, points, format);
  if (rc != PS_OK) { ps_bases_free(b); return rc; }
  *out = b;
  return PS_OK;
}

// One segment of a batched MSM: `n` scalars at `scalars` against points [first, first + n) of `b`, summed
// into output `set`.
struct SegSpec { const ps_bases* b; size_t first; const uint32_t* scalars; size_t n; int mont; int set; };

// Runs `nseg` segments over `nsets` outputs as ONE Pippenger pipeline (shared digit pass, sort, accumulation
// and tail).  Segments that write the same output must name the same base set.  All base sets of a batch
// must agree on the window geometry: key loaders give every base set of a key the same window.
template <class F>
int msm_batch(ps_ctx* ctx, const SegSpec* segs, int nseg, int nsets, XYZZ<F>* d_out) {
  if (nseg < 1 || nseg > MSM_MAX_SEG || nsets < 1 || nsets > MSM_MAX_SEG) return PS_ERR_ARG;
  MsmPlan p;
  memset(&p, 0, sizeof p);
  size_t total = 0;
  const ps_bases* of_set[MSM_MAX_SEG] = {nullptr};
  for (int k = 0; k < nseg; k++) {
    const SegSpec& sg = segs[k];
    if (!sg.b || sg.set < 0 || sg.set >= nsets || sg.b->group != PointBytes<F>::GROUP) return PS_ERR_ARG;
    if (sg.first + sg.n > sg.b->n) return PS_ERR_LENGTH;
    if (of_set[sg.set] && of_set[sg.set] != sg.b) return PS_ERR_ARG;
    of_set[sg.set] = sg.b;
    total += sg.n;
  }
  if (total >= 0xFFFFFFFFull) return PS_ERR_UNSUPPORTED;
  // one pipeline needs one table allocation and one window geometry; base sets loaded separately run one after the other
  const void* slab = nullptr;
  int c = 0, T = 0;
  bool uniform = true;
  for (int s = 0; s < nsets; s++) {
    const ps_bases* b = of_set[s];
    if (!b) continue;
    if (T == 0) { c = b->c; T = b->T; slab = b->slab; }
    else if (b->c != c || b->T != T || b->slab != slab) uniform = false;
  }
  if (!uniform) {
    for (int s = 0; s < nsets; s++) {
      SegSpec sub[MSM_MAX_SEG];
      int cnt = 0;
      for (int k = 0; k < nseg; k++)
        if (segs[k].set == s) { sub[cnt] = segs[k]; sub[cnt].set = 0; cnt++; }
      if (cnt) PS_TRY(msm_batch<F>(ctx, sub, cnt, 1, d_out + s));
      else PS_TRY(dev_memset(d_out + s, 0, sizeof(XYZZ<F>), ctx->stream));
    }
    return PS_OK;
  }
  if (T == 0) { c = 0; T = 1; }
  if (c == 0) c = msm_pick_window(total ? total : 1);
  p.c = c; p.W = msm_windows(c); p.T = T; p.S = (p.W + T - 1) / T; p.D = 1u << (c - 1);
  p.total = (uint32_t)total; p.nseg = nseg; p.nsets = nsets;
  uint32_t start = 0;
  for (int k = 0; k < nseg; k++) {
    const SegSpec& sg = segs[k];
    p.seg[k].scalars = sg.scalars; p.seg[k].n = (uint32_t)sg.n; p.seg[k].start = start;
    p.seg[k].first = (uint32_t)sg.first; p.seg[k].set = (uint32_t)sg.set; p.seg[k].mont = (uint32_t)sg.mont;
    start += (uint32_t)sg.n;
  }
  for (int s = 0; s < nsets; s++) {
    const ps_bases* b = of_set[s];
    p.nbase[s] = b ? (uint32_t)b->n : 0;
    p.toff[s] = b ? (uint32_t)(((const char*)b->tab - (const char*)slab) / sizeof(Affine<F>)) : 0;
  }
  return GroupOps<F>::msm_batch(ctx, p, (const Affine<F>*)slab, d_out);
}

template <class F>
int msm_on_bases(ps_ctx* ctx, const ps_bases* b, size_t first, const uint32_t* d_scalars, size_t n, int mont, XYZZ<F>* d_out) {
  if (first + n > b->n) return PS_ERR_LENGTH;
  SegSpec sg{b, first, d_scalars, n, mont, 0};
  return msm_batch<F>(ctx, &sg, 1, 1, d_out);
}

template <class F>
int encode_points(ps_ctx* ctx, const XYZZ<F>* d_pts, size_t count, uint8_t* host_out) {
  size_t per = PointBytes<F>::COMP;
  uint8_t* d_bytes = ctx->arena.take<uint8_t>(count * per);
  if (!d_bytes) return PS_ERR_ALLOC;
  PS_TRY(GroupOps<F>::encode_xyzz(ctx, d_pts, count, (int)PS_FMT_COMPRESSED, d_bytes));
  PS_TRY(dev_d2h(host_out, d_bytes, count * per, ctx->stream));
  return PS_OK;
}

// the same into the context's page-locked staging area (offset in bytes): does not block the host
template <class F>
int encode_points_staged(ps_ctx* ctx, const XYZZ<F>* d_pts, size_t count, size_t stage_off) {
  if (stage_off + count * PointBytes<F>::COMP > ps_ctx::H_STAGE_BYTES) return PS_ERR_ARG;
  return encode_points<F>(ctx, d_pts, count, ctx->h_stage + stage_off);
}

// concatenates host point arrays and loads them into the allocated base set `b` (sum of counts == b->n)
template <class F>
int bases_concat_into(ps_ctx* ctx, ps_bases* b, int format, const uint8_t* const* parts, const size_t* counts, int nparts) {
  size_t per = point_bytes(PointBytes<F>::GROUP, format), total = 0;
  for (int i = 0; i < nparts; i++) total += counts[i];
  if (total != b->n) return PS_ERR_ARG;
  std::vector<uint8_t> buf(total * per);
  size_t o = 0;
  for (int i = 0; i < nparts; i++) {
    if (counts[i] && !parts[i]) return PS_ERR_ARG;
    memcpy(buf.data() + o, parts[i], counts[i] * per);
    o += counts[i] * per;
  }
  return bases_fill_t<F>(ctx, b, buf.data(), format);
}

// allocates the three base sets of a Groth16 key: A and C carved out of one G1 slab, B (G2) on its own
int g16_key_alloc(ps_g16_key* k, size_t nA, size_t nB, size_t nC, int window_g1, int window_g2) {
  const size_t g1counts[2] = {nA, nC};
  ps_bases* g1[2] = {nullptr, nullptr};
  PS_TRY(bases_alloc_slab(PS_G1, g1counts, 2, window_g1, &k->slab_g1, g1));
  k->A = g1[0]; k->C = g1[1];
  void* slab_b = nullptr;
  PS_TRY(bases_alloc_slab(PS_G2, &nB, 1, window_g2, &slab_b, &k->B));
  k->B->owns = true;    // a one-set slab: the base set owns its allocation
  return PS_OK;
}
// the eight base sets of a PHGR13 evaluation key: the seven G1 ones in one slab
int phgr13_key_alloc(ps_ctx* ctx, ps_phgr13_key* k, size_t n_gates, size_t n_mid) {
  const size_t counts[7] = {n_gates - 1, n_mid, n_mid, n_mid, n_mid, n_mid, 3 * n_mid};
  // the seven G1 sums of a proof run as one batch (pinochio.go:218-242 sums the same solution[diff:] against eight base
  // vectors); wss (G2) on its own
  PS_TRY(bases_alloc_slab(PS_G1, counts, 7, batch_window(ctx, n_gates - 1 + 8 * n_mid, 7), &k->slab_g1, k->g1));
  void* slab_w = nullptr;
  PS_TRY(bases_alloc_slab(PS_G2, &n_mid, 1, batch_window(ctx, n_mid, 1), &slab_w, &k->ws));
  k->ws->owns = true;
  return PS_OK;
}

}  // namespace

namespace ps {
// window of a batch of `nsets` MSMs over `total_points` points in all (per shard): every set pays its own bucket
// merge + reduction, the mixed additions are shared (same model as msm_pick_window_full, which is the case nsets = 1)
int batch_window(ps_ctx* ctx, size_t total_points, int nsets) {
  const size_t shards = (size_t)(ctx->msm_shards > 0 ? ctx->msm_shards : 1);
  const double n = (double)(total_points / shards + 1), bucket_cost = (double)ctx->msm_bucket_cost * (nsets > 0 ? nsets : 1);
  int best = 4; double best_cost = 1e300;
  for (int c = 4; c <= 24; c++) {
    double W = msm_windows(c);
    if (n * W >= 2.0e9) continue;
    double cost = n * W * 10.0 + (double)(1u << (c - 1)) * bucket_cost;
    if (cost < best_cost) { best_cost = cost; best = c; }
  }
  return best;
}

template <class F>
int msm_rows(ps_ctx* ctx, const ps_bases* b, const uint32_t* d_scalars, size_t rows, int mont, XYZZ<F>* d_out) {
  if (!b || b->group != PointBytes<F>::GROUP) return PS_ERR_ARG;
  if (rows == 0) return PS_OK;
  const size_t n = b->n;
  if (n == 0) return dev_memset(d_out, 0, rows * sizeof(XYZZ<F>), ctx->stream);
  // every row has its own bucket sets, so a window without precomputed tables is chosen as for one row
  const int c = b->c ? b->c : msm_pick_window(n), W = msm_windows(c), T = b->T, S = (W + T - 1) / T;
  // rows per pipeline: entry positions and bucket indices of one pipeline stay below 2^31
  const size_t lim = 0x7FFFFFFFull, per = std::max((size_t)n * W, (size_t)S << (c - 1));
  if (per > lim) return PS_ERR_UNSUPPORTED;
  const size_t cap = lim / per;
  for (size_t r0 = 0; r0 < rows; r0 += cap) {
    const size_t cnt = std::min(cap, rows - r0);
    MsmPlan p;
    memset(&p, 0, sizeof p);
    p.c = c; p.W = W; p.T = T; p.S = S; p.D = 1u << (c - 1);
    p.total = (uint32_t)(cnt * n); p.nseg = 1; p.nsets = (int)cnt; p.row_len = (uint32_t)n;
    p.seg[0].scalars = d_scalars + r0 * n * 8; p.seg[0].n = p.total; p.seg[0].mont = (uint32_t)mont;
    p.nbase[0] = (uint32_t)n;
    p.toff[0] = (uint32_t)(((const char*)b->tab - (const char*)b->slab) / sizeof(Affine<F>));
    PS_TRY(GroupOps<F>::msm_batch(ctx, p, (const Affine<F>*)b->slab, d_out + r0));
  }
  return PS_OK;
}
template int msm_rows<Fp>(ps_ctx*, const ps_bases*, const uint32_t*, size_t, int, XYZZ<Fp>*);
template int msm_rows<Fp2>(ps_ctx*, const ps_bases*, const uint32_t*, size_t, int, XYZZ<Fp2>*);
}  // namespace ps

extern "C" {

const char* ps_strerror(int status) {
  switch (status) {
    case PS_OK: return "ok";
    case PS_ERR_ARG: return "bad argument";
    case PS_ERR_LENGTH: return "mismatch of length between poly and blinded eval points";
    case PS_ERR_REMAINDER: return "apocalypse";
    case PS_ERR_ENCODING: return "bad scalar or point encoding";
    case PS_ERR_CUDA: return "CUDA error";
    case PS_ERR_ALLOC: return "out of memory";
    case PS_ERR_UNSUPPORTED: return "unsupported";
    default: return "unknown status";
  }
}

const char* ps_version(void) {
#if PS_GPU
  return "playsnark_b200 0.1 (sm_100a)";
#else
  return "playsnark_b200 0.1 (HOST EMULATION - tests only)";
#endif
}

uint64_t ps_launch_count(void) { return launch_counter(); }

int ps_ctx_create(int device, ps_ctx** out) {
  if (!out) return PS_ERR_ARG;
  ps_ctx* ctx = new (std::nothrow) ps_ctx();
  if (!ctx) return PS_ERR_ALLOC;
  ctx->device = device;
  int rc = PS_OK;
#if PS_GPU
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) {
    fprintf(stderr, "playsnark_b200: no CUDA device %d (found %d); there is no CPU fallback\n", device, count);
    delete ctx;
    return PS_ERR_CUDA;
  }
  // every failure below goes through ps_ctx_destroy, which releases whatever has been created so far
  auto init = [&]() -> int {
    PS_CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    PS_CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    ctx->sm_count = prop.multiProcessorCount;
    cudaStream_t st;
    PS_CUDA_TRY(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    ctx->stream = st;
    ctx->own_stream = true;
    // The secondary stream carries the G2 sum of a proof next to the G1 batch.  At HIGH priority its blocks are placed
    // first: the G2 accumulation runs ahead and its latency-bound tail (tiny grids) then slips in between the blocks of
    // the G1 accumulation instead of queueing behind them.  PLAYSNARK_B200_STREAM2_PRIO=0 keeps the default priority (A/B).
    cudaStream_t st2;
    int prio_lo = 0, prio_hi = 0;
    PS_CUDA_TRY(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    const char* pe = getenv("PLAYSNARK_B200_STREAM2_PRIO");
    const int prio = (pe && pe[0] == '0') ? prio_lo : prio_hi;
    PS_CUDA_TRY(cudaStreamCreateWithPriority(&st2, cudaStreamNonBlocking, prio));
    ctx->stream2 = st2;
    cudaEvent_t e;
    PS_CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); ctx->ev_fork = e;
    PS_CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); ctx->ev_join = e;
    for (int i = 0; i < 5; i++) { PS_CUDA_TRY(cudaEventCreate(&e)); ctx->ev[i] = e; }
    for (int i = 0; i < 6; i++) { PS_CUDA_TRY(cudaEventCreate(&e)); ctx->evp[i] = e; }
    for (int i = 0; i < 9; i++) { PS_CUDA_TRY(cudaEventCreate(&e)); ctx->evv[i] = e; }
    return PS_OK;
  };
  rc = init();
#endif
  ctx->arena.stream = ctx->stream;
  ctx->arena2.stream = ctx->stream2;
  if (rc == PS_OK) {
    void* hp = nullptr;
    rc = ps_host_alloc(ps_ctx::H_STAGE_BYTES, &hp);
    ctx->h_stage = (uint8_t*)hp;
  }
  if (rc != PS_OK) { ps_ctx_destroy(ctx); return rc; }
  *out = ctx;
  return PS_OK;
}

int ps_ctx_set_stream(ps_ctx* ctx, void* cuda_stream) {
  if (!ctx) return PS_ERR_ARG;
#if PS_GPU
  PS_TRY(dev_sync(ctx->stream));
  if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
  ctx->stream = (cudaStream_t)cuda_stream;
  ctx->own_stream = false;
  ctx->arena.stream = ctx->stream;
#else
  (void)cuda_stream;
#endif
  return PS_OK;
}

int ps_ctx_set_option(ps_ctx* ctx, const char* name, int value) {
  if (!ctx || !name) return PS_ERR_ARG;
  if (!strcmp(name, "interp_fused")) {
    if (value != 0 && value != 1) return PS_ERR_ARG;
    ctx->interp_fused = value;
    return PS_OK;
  }
  if (!strcmp(name, "subgroup_check")) {
    if (value != 0 && value != 1) return PS_ERR_ARG;
    ctx->subgroup_check = value;
    return PS_OK;
  }
  if (!strcmp(name, "msm_shards")) {
    if (value < 1 || value > 1024) return PS_ERR_ARG;
    ctx->msm_shards = value;
    return PS_OK;
  }
  if (!strcmp(name, "msm_bucket_cost")) {
    if (value < 1 || value > 100000) return PS_ERR_ARG;
    ctx->msm_bucket_cost = value;
    return PS_OK;
  }
  if (!strcmp(name, "msm_scatter")) {
    if (value < 0 || value > 2) return PS_ERR_ARG;
    ctx->msm_scatter = value;
    return PS_OK;
  }
  if (!strcmp(name, "msm_wave_floor")) {
    if (value != 0 && value != 1) return PS_ERR_ARG;
    ctx->msm_wave_floor = value;
    return PS_OK;
  }
  if (!strcmp(name, "msm_team")) {
    if (value != 0 && value != 1) return PS_ERR_ARG;
    ctx->msm_team = value;
    return PS_OK;
  }
  return PS_ERR_ARG;
}

int ps_ctx_sync(ps_ctx* ctx) { return ctx ? dev_sync(ctx->stream) : PS_ERR_ARG; }

void ps_ctx_destroy(ps_ctx* ctx) {
  if (!ctx) return;
  if (ctx->stream) dev_sync(ctx->stream);
  if (ctx->stream2) dev_sync(ctx->stream2);
  ctx->arena.release();
  ctx->arena2.release();
  for (auto& t : ctx->ntt_cache) t.release();
  dev_free(ctx->fixed_base[0]);
  dev_free(ctx->fixed_base[1]);
  ps_host_free(ctx->h_stage);
#if PS_GPU
  for (int i = 0; i < 5; i++) if (ctx->ev[i]) cudaEventDestroy((cudaEvent_t)ctx->ev[i]);
  for (int i = 0; i < 6; i++) if (ctx->evp[i]) cudaEventDestroy((cudaEvent_t)ctx->evp[i]);
  for (int i = 0; i < 9; i++) if (ctx->evv[i]) cudaEventDestroy((cudaEvent_t)ctx->evv[i]);
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
  if (ctx->ev_fork) cudaEventDestroy((cudaEvent_t)ctx->ev_fork);
  if (ctx->ev_join) cudaEventDestroy((cudaEvent_t)ctx->ev_join);
#endif
  delete ctx;
}

// ---- bases ------------------------------------------------------------------------------------------
int ps_bases_load(ps_ctx* ctx, int group, const uint8_t* points, size_t n, int format, int window_bits,
                  int precompute_tables, ps_bases** out) {
  if (!out || (n && !points) || (format != PS_FMT_COMPRESSED && format != PS_FMT_AFFINE)) return PS_ERR_ARG;
  PS_TRY(begin_call(ctx));
  if (group == PS_G1) return bases_load_t<Fp>(ctx, points, n, format, window_bits, precompute_tables, out);
  if (group == PS_G2) return bases_load_t<Fp2>(ctx, points, n, format, window_bits, precompute_tables, out);
  return PS_ERR_ARG;
}

size_t ps_bases_len(const ps_bases* b) { return b ? b->n : 0; }

int ps_bases_info(const ps_bases* b, int out[4]) {
  if (!b || !out) return PS_ERR_ARG;
  int c = b->c ? b->c : msm_pick_window(b->n ? b->n : 1);
  out[0] = c; out[1] = msm_windows(c); out[2] = b->T; out[3] = b->group;
  return PS_OK;
}

void ps_bases_free(ps_bases* b) {
  if (!b) return;
  if (b->owns) dev_free(b->tab);
  delete b;
}

int ps_bases_from_scalars(ps_ctx* ctx, int group, const uint8_t* scalars_be, size_t n, int window_bits,
                          int precompute_tables, ps_bases** out) {
  if (!out || (n && !scalars_be) || (group != PS_G1 && group != PS_G2)) return PS_ERR_ARG;
  PS_TRY(begin_call(ctx));
  ps_bases* b = nullptr;
  PS_TRY(bases_alloc(group, n, window_bits, precompute_tables, ctx->msm_shards, ctx->msm_bucket_cost, &b));
  uint32_t *d_sc = nullptr, *d_err = nullptr;
  int rc = stage_scalars(ctx, scalars_be, n, 0, &d_sc, &d_err);
  if (rc == PS_OK) {
    if (group == PS_G1) {
      rc = GroupOps<Fp>::from_scalars(ctx, d_sc, n, (G1Affine*)b->tab);
      if (rc == PS_OK) rc = GroupOps<Fp>::tables_finish(ctx, (G1Affine*)b->tab, b->n, b->c, b->T);
    } else {
      rc = GroupOps<Fp2>::from_scalars(ctx, d_sc, n, (G2Affine*)b->tab);
      if (rc == PS_OK) rc = GroupOps<Fp2>::tables_finish(ctx, (G2Affine*)b->tab, b->n, b->c, b->T);
    }
  }
  if (rc == PS_OK) rc = check_err_flag(ctx, d_err, PS_ERR_ENCODING);
  if (rc != PS_OK) { ps_bases_free(b); return rc; }
  *out = b;
  return PS_OK;
}

int ps_bases_export(ps_ctx* ctx, const ps_bases* b, size_t first, size_t count, int format, uint8_t* out) {
  if (!b || !out || first + count > b->n || (format != PS_FMT_COMPRESSED && format != PS_FMT_AFFINE)) return PS_ERR_ARG;
  PS_TRY(begin_call(ctx));
  size_t per = point_bytes(b->group, format);
  uint8_t* d_bytes = ctx->arena.take<uint8_t>(count * per);
  if (!d_bytes) return PS_ERR_ALLOC;
  if (b->group == PS_G1) PS_TRY(GroupOps<Fp>::encode_affine(ctx, (const G1Affine*)b->tab + first, count, format, d_bytes));
  else PS_TRY(GroupOps<Fp2>::encode_affine(ctx, (const G2Affine*)b->tab + first, count, format, d_bytes));
  PS_TRY(dev_d2h(out, d_bytes, count * per, ctx->stream));
  return dev_sync(ctx->stream);
}

// ---- MSM --------------------------------------------------------------------------------------------
int ps_msm(ps_ctx* ctx, const ps_bases* b, const uint8_t* scalars_be, size_t n, uint8_t* out) {
  if (!b || !out || (n && !scalars_be)) return PS_ERR_ARG;
  if (n != b->n) return PS_ERR_LENGTH;
  PS_TRY(begin_call(ctx));
  uint32_t *d_sc = nullptr, *d_err = nullptr;
  PS_TRY(stage_scalars(ctx, scalars_be, n, 0, &d_sc, &d_err));
  if (b->group == PS_G1) {
    G1XYZZ* d_res = ctx->arena.take<G1XYZZ>(1);
    if (!d_res) return PS_ERR_ALLOC;
    PS_TRY(msm_on_bases<Fp>(ctx, b, 0, d_sc, n, 0, d_res));
    PS_TRY(encode_points<Fp>(ctx, d_res, 1, out));
  } else {
    G2XYZZ* d_res = ctx->arena.take<G2XYZZ>(1);
    if (!d_res) return PS_ERR_ALLOC;
    PS_TRY(msm_on_bases<Fp2>(ctx, b, 0, d_sc, n, 0, d_res));
    PS_TRY(encode_points<Fp2>(ctx, d_res, 1, out));
  }
  return check_err_flag(ctx, d_err, PS_ERR_ENCODING);
}

int ps_msm_rows(ps_ctx* ctx, const ps_bases* b, const uint8_t* scalars_be, size_t n, size_t rows, uint8_t* out) {
  if (!b || (rows && !out) || (rows && n && !scalars_be)) return PS_ERR_ARG;
  if (n != b->n) return PS_ERR_LENGTH;
  if (n && rows > ((size_t)1 << 40) / n) return PS_ERR_UNSUPPORTED;
  PS_TRY(begin_call(ctx));
  if (rows == 0) return PS_OK;
  uint32_t *d_sc = nullptr, *d_err = nullptr;
  PS_TRY(stage_scalars(ctx, scalars_be, rows * n, 0, &d_sc, &d_err));
  if (b->group == PS_G1) {
    G1XYZZ* d_res = ctx->arena.take<G1XYZZ>(rows);
    if (!d_res) return PS_ERR_ALLOC;
    PS_TRY(msm_rows<Fp>(ctx, b, d_sc, rows, 0, d_res));
    PS_TRY(encode_points<Fp>(ctx, d_res, rows, out));
  } else {
    G2XYZZ* d_res = ctx->arena.take<G2XYZZ>(rows);
    if (!d_res) return PS_ERR_ALLOC;
    PS_TRY(msm_rows<Fp2>(ctx, b, d_sc, rows, 0, d_res));
    PS_TRY(encode_points<Fp2>(ctx, d_res, rows, out));
  }
  return check_err_flag(ctx, d_err, PS_ERR_ENCODING);
}

int ps_msm_device(ps_ctx* ctx, const ps_bases* b, size_t first, const void* d_scalars_le, size_t n, void* d_out_xyzz) {
  if (!b || !d_out_xyzz || (n && !d_scalars_le)) return PS_ERR_ARG;
  PS_TRY(begin_call(ctx));
  if (b->group == PS_G1) return msm_on_bases<Fp>(ctx, b, first, (const uint32_t*)d_scalars_le, n, 0, (G1XYZZ*)d_out_xyzz);
  return msm_on_bases<Fp2>(ctx, b, first, (const uint32_t*)d_scalars_le, n, 0, (G2XYZZ*)d_out_xyzz);
}

/* the same with the scalars in Montgomery form (what ps_fr_upload leaves on the device) */
int ps_msm_device_mont(ps_ctx* ctx, const ps_bases* b, size_t first, const void* d_scalars_mont, size_t n, void* d_out_xyzz) {
  if (!b || !d_out_xyzz || (n && !d_scalars_mont)) return PS_ERR_ARG;
  PS_TRY(begin_call(ctx));
  if (b->group == PS_G1) return msm_on_bases<Fp>(ctx, b, first, (const uint32_t*)d_scalars_mont, n, 1, (G1XYZZ*)d_out_xyzz);
  return msm_on_bases<Fp2>(ctx, b, first, (const uint32_t*)d_scalars_mont, n, 1, (G2XYZZ*)d_out_xyzz);
}

int ps_msm_combine(ps_ctx* ctx, int group, const void* d_partials_xyzz, size_t count, uint8_t* out) {
  if (!d_partials_xyzz || !out || (group != PS_G1 && group != PS_G2)) return PS_ERR_ARG;
  PS_TRY(begin_call(ctx));
  if (group == PS_G1) {
    G1XYZZ* d_res = ctx->arena.take<G1XYZZ>(1);
    if (!d_res) return PS_ERR_ALLOC;
    PS_TRY(GroupOps<Fp>::sum_points(ctx, (const G1XYZZ*)d_partials_xyzz, (uint32_t)count, d_res));
    PS_TRY(encode_points<Fp>(ctx, d_res, 1, out));
  } else {
    G2XYZZ* d_res = ctx->arena.take<G2XYZZ>(1);
    if (!d_res) return PS_ERR_ALLOC;
    PS_TRY(GroupOps<Fp2>::sum_points(ctx, (const G2XYZZ*)d_partials_xyzz, (uint32_t)count, d_res));
    PS_TRY(encode_points<Fp2>(ctx, d_res, 1, out));
  }
  return dev_sync(ctx->stream);
}

int ps_last_msm_timing(ps_ctx* ctx, float out_ms[5]) {
  if (!ctx || !out_ms) return PS_ERR_ARG;
  for (int i = 0; i < 5; i++) out_ms[i] = 0.f;
#if PS_GPU
  if (!ctx->ev_valid) return PS_ERR_ARG;
  PS_CUDA_TRY(cudaEventSynchronize((cudaEvent_t)ctx->ev[4]));
  for (int i = 0; i < 4; i++)
    PS_CUDA_TRY(cudaEventElapsedTime(&out_ms[i], (cudaEvent_t)ctx->ev[i], (cudaEvent_t)ctx->ev[i + 1]));
  PS_CUDA_TRY(cudaEventElapsedTime(&out_ms[4], (cudaEvent_t)ctx->ev[0], (cudaEvent_t)ctx->ev[4]));
#endif
  return PS_OK;
}

int ps_last_prove_timing(ps_ctx* ctx, float out_ms[6]) {
  if (!ctx || !out_ms) return PS_ERR_ARG;
  for (int i = 0; i < 6; i++) out_ms[i] = 0.f;
#if PS_GPU
  if (!ctx->evp_valid) return PS_ERR_ARG;
  PS_CUDA_TRY(cudaEventSynchronize((cudaEvent_t)ctx->evp[5]));
  for (int i = 0; i < 5; i++)
    PS_CUDA_TRY(cudaEventElapsedTime(&out_ms[i], (cudaEvent_t)ctx->evp[i], (cudaEvent_t)ctx->evp[i + 1]));
  PS_CUDA_TRY(cudaEventElapsedTime(&out_ms[5], (cudaEvent_t)ctx->evp[0], (cudaEvent_t)ctx->evp[5]));
#endif
  return PS_OK;
}

int ps_last_verify_batch_timing(ps_ctx* ctx, float out_ms[9]) {
  if (!ctx || !out_ms) return PS_ERR_ARG;
  for (int i = 0; i < 9; i++) out_ms[i] = 0.f;
#if PS_GPU
  if (!ctx->evv_valid) return PS_ERR_ARG;
  PS_CUDA_TRY(cudaEventSynchronize((cudaEvent_t)ctx->evv[8]));
  for (int i = 0; i < 8; i++)
    PS_CUDA_TRY(cudaEventElapsedTime(&out_ms[i], (cudaEvent_t)ctx->evv[i], (cudaEvent_t)ctx->evv[i + 1]));
  PS_CUDA_TRY(cudaEventElapsedTime(&out_ms[8], (cudaEvent_t)ctx->evv[0], (cudaEvent_t)ctx->evv[8]));
#endif
  return PS_OK;
}

// ---- Groth16 ------------------------------------------------------------------------------------------
// The proof elements are assembled as three MSMs over concatenated base sets (same group elements as
// groth16.go:146-200, which adds the pieces one scalar multiplication at a time):
//   A = <[a | r | 1],            [Xi  | Delta  | Alpha]>
//   B = <[b | s | 1],            [Xi2 | Delta2 | Beta2]>
//   C = <[w_nio | h | s a + r b | s | r | r s], [NioLP | XiT | Xi | Alpha | Beta | Delta]>
// using  s A + r B1 - r s Delta = sum_k (s a_k + r b_k) Xi_k + s Alpha + r Beta + r s Delta.
// A and C (both G1) run as one batched pipeline; B (G2) runs concurrently on the second stream.
int ps_g16_key_load(ps_ctx* ctx, size_t n_gates, size_t n_nio, int format, const uint8_t* xi, const uint8_t* xi2,
                    const uint8_t* xit, const uint8_t* niolp, const uint8_t* alpha, const uint8_t* beta,
                    const uint8_t* delta, const uint8_t* beta2, const uint8_t* delta2, ps_g16_key** key) {
  if (!key || !xi || !xi2 || !xit || (n_nio && !niolp) || !alpha || !beta || !delta || !beta2 || !delta2 || n_gates < 2)
    return PS_ERR_ARG;
  if (format != PS_FMT_COMPRESSED && format != PS_FMT_AFFINE) return PS_ERR_ARG;
  PS_TRY(begin_call(ctx));
  ps_g16_key* k = new (std::nothrow) ps_g16_key();
  if (!k) return PS_ERR_ALLOC;
  k->n = n_gates; k->n_nio = n_nio;
  const uint8_t* pa[3] = {xi, delta, alpha};
  const size_t ca[3] = {n_gates, 1, 1};
  const uint8_t* pb[3] = {xi2, delta2, beta2};
  const uint8_t* pc[6] = {niolp, xit, xi, alpha, beta, delta};
  const size_t cc[6] = {n_nio, n_gates - 1, n_gates, 1, 1, 1};
  // A and C share a pipeline (one window for both); B has its own
  int rc = g16_key_alloc(k, n_gates + 2, n_gates + 2, n_nio + (n_gates - 1) + n_gates + 3,
                         batch_window(ctx, 3 * n_gates + n_nio + 4, 2), batch_window(ctx, n_gates + 2, 1));
  if (rc == PS_OK) rc = bases_concat_into<Fp>(ctx, k->A, format, pa, ca, 3);
  if (rc == PS_OK) rc = ctx->arena.reset();
  if (rc == PS_OK) rc = bases_concat_into<Fp2>(ctx, k->B, format, pb, ca, 3);
  if (rc == PS_OK) rc = ctx->arena.reset();
  if (rc == PS_OK) rc = bases_concat_into<Fp>(ctx, k->C, format, pc, cc, 6);
  if (rc != PS_OK) { ps_g16_key_free(k); return rc; }
  *key = k;
  return PS_OK;
}

void ps_g16_key_free(ps_g16_key* key) {
  if (!key) return;
  ps_bases_free(key->A); ps_bases_free(key->B); ps_bases_free(key->C);
  dev_free(key->slab_g1);
  delete key;
}

int ps_g16_prove(ps_ctx* ctx, const ps_g16_key* key, const ps_qap* qap, const uint8_t* witness_be, const uint8_t* r_be,
                 const uint8_t* s_be, uint8_t* outA, uint8_t* outB, uint8_t* outC, uint8_t* out_h) {
  if (!key || !qap || !witness_be || !r_be || !s_be || !outA || !outB || !outC) return PS_ERR_ARG;
  PS_TRY(begin_call(ctx));
  G16Scalars sc;
  ctx->evp_valid = false;
  PS_TRY(ctx_prove_event(ctx, 0));
  PS_TRY(g16_build_scalars(ctx, key, qap, witness_be, r_be, s_be, &sc));
  PS_TRY(ctx_prove_event(ctx, 1));
  G1XYZZ* resG1 = ctx->arena.take<G1XYZZ>(2);
  G2XYZZ* resG2 = ctx->arena.take<G2XYZZ>(1);
  if (!resG1 || !resG2) return PS_ERR_ALLOC;
  // the G2 MSM is independent of the two G1 ones: it runs on the secondary stream so that its serial
  // tails and its register-bound accumulate kernel overlap with the G1 work
  PS_TRY(ctx_fork(ctx));
  ForkGuard fg(ctx);
  {
    SecondaryScope scope(ctx);
    PS_TRY(msm_on_bases<Fp2>(ctx, key->B, 0, (const uint32_t*)sc.scB, sc.nB, 1, resG2));
    PS_TRY(encode_points_staged<Fp2>(ctx, resG2, 1, 96));   // its inversion chain overlaps the G1 work too
  }
  const SegSpec g1segs[2] = {{key->A, 0, (const uint32_t*)sc.scA, sc.nA, 1, 0}, {key->C, 0, (const uint32_t*)sc.scC, sc.nC, 1, 1}};
  PS_TRY(msm_batch<Fp>(ctx, g1segs, 2, 2, resG1));
  PS_TRY(ctx_prove_event(ctx, 2));
  PS_TRY(ctx_prove_event(ctx, 3));
  PS_TRY(encode_points_staged<Fp>(ctx, resG1, 2, 0));
  PS_TRY(ctx_prove_event(ctx, 4));
  PS_TRY(fg.join());
  PS_TRY(ctx_prove_event(ctx, 5));
  ctx->evp_valid = true;
  if (out_h) PS_TRY(export_fr(ctx, sc.qb.h, qap->n - 1, out_h));
  PS_TRY(check_err_flag(ctx, sc.qb.enc_err, PS_ERR_ENCODING));
  PS_TRY(check_err_flag(ctx, sc.qb.flag, PS_ERR_REMAINDER));   // synchronises the primary stream, which has joined the second
  memcpy(outA, ctx->h_stage, 48);
  memcpy(outC, ctx->h_stage + 48, 48);
  memcpy(outB, ctx->h_stage + 96, 96);
  return PS_OK;
}

extern "C++" {
namespace ps {
int g16_key_load_slice(ps_ctx* ctx, const KeySlice& sl, int format, int window_g1, int window_g2, const uint8_t* xi, const uint8_t* xi2,
                       const uint8_t* xit, const uint8_t* niolp, const uint8_t* alpha, const uint8_t* beta, const uint8_t* delta,
                       const uint8_t* beta2, const uint8_t* delta2, ps_g16_key** key) {
  if (!key || sl.x_hi < sl.x_lo || sl.t_hi < sl.t_lo || sl.n_hi < sl.n_lo) return PS_ERR_ARG;
  if (format != PS_FMT_COMPRESSED && format != PS_FMT_AFFINE) return PS_ERR_ARG;
  PS_TRY(begin_call(ctx));
  ps_g16_key* k = new (std::nothrow) ps_g16_key();
  if (!k) return PS_ERR_ALLOC;
  const size_t g1 = point_bytes(PS_G1, format), g2 = point_bytes(PS_G2, format);
  const size_t nx = sl.x_hi - sl.x_lo, nt = sl.t_hi - sl.t_lo, nn = sl.n_hi - sl.n_lo, one = sl.consts ? 1 : 0;
  k->n = nx; k->n_nio = nn;   // sizes of this slice (the orchestration keeps the global ones)
  const uint8_t* pa[3] = {xi + sl.x_lo * g1, delta, alpha};
  const size_t ca[3] = {nx, one, one};
  const uint8_t* pb[3] = {xi2 + sl.x_lo * g2, delta2, beta2};
  const uint8_t* pc[6] = {niolp ? niolp + sl.n_lo * g1 : niolp, xit + sl.t_lo * g1, xi + sl.x_lo * g1, alpha, beta, delta};
  const size_t cc[6] = {nn, nt, nx, one, one, one};
  int rc = g16_key_alloc(k, nx + 2 * one, nx + 2 * one, nn + nt + nx + 3 * one, window_g1, window_g2);
  if (rc == PS_OK) rc = bases_concat_into<Fp>(ctx, k->A, format, pa, ca, 3);
  if (rc == PS_OK) rc = ctx->arena.reset();
  if (rc == PS_OK) rc = bases_concat_into<Fp2>(ctx, k->B, format, pb, ca, 3);
  if (rc == PS_OK) rc = ctx->arena.reset();
  if (rc == PS_OK) rc = bases_concat_into<Fp>(ctx, k->C, format, pc, cc, 6);
  if (rc != PS_OK) { ps_g16_key_free(k); return rc; }
  *key = k;
  return PS_OK;
}

int g16_slice_msm_all(ps_ctx* ctx, const ps_g16_key* key, const KeySlice& sl, const Fr* scA, const Fr* scB, const Fr* scC,
                      void* d_partials, const std::function<int()>& before_g1) {
  PS_TRY(begin_call(ctx));
  uint8_t* out = (uint8_t*)d_partials;  // [A: 192 B | C: 192 B | B: 384 B | 192 B left zero (infinity)]
  const size_t nx = sl.x_hi - sl.x_lo, nt = sl.t_hi - sl.t_lo, nn = sl.n_hi - sl.n_lo, k3 = sl.consts ? 3 : 0, k2 = sl.consts ? 2 : 0;
  PS_TRY(ctx_fork(ctx));
  ForkGuard fg(ctx);
  {
    SecondaryScope scope(ctx);
    PS_TRY(msm_on_bases<Fp2>(ctx, key->B, 0, (const uint32_t*)scB, nx + k2, 0, (G2XYZZ*)(out + 384)));
  }
  if (before_g1) PS_TRY(before_g1());   // e.g. the primary stream starts waiting for h here, with B_d already under way
  // scC = [w_nio | h | s a + r b | s r rs] against C_d = [NioLP | XiT | Xi | Alpha Beta Delta]: one contiguous segment
  const SegSpec segs[2] = {{key->A, 0, (const uint32_t*)scA, nx + k2, 0, 0},
                           {key->C, 0, (const uint32_t*)scC, nn + nt + nx + k3, 0, 1}};
  PS_TRY(msm_batch<Fp>(ctx, segs, 2, 2, (G1XYZZ*)out));
  PS_TRY(dev_memset(out + 768, 0, 192, ctx->stream));
  return fg.join();
}

int msm_partial_host_scalars(ps_ctx* ctx, const ps_bases* b, const uint8_t* scalars_be, size_t n, void* d_out_xyzz, uint32_t** d_err_out) {
  if (!b || n != b->n) return PS_ERR_LENGTH;
  PS_TRY(begin_call(ctx));
  uint32_t* d_sc = nullptr;
  PS_TRY(stage_scalars(ctx, scalars_be, n, 0, &d_sc, d_err_out));
  if (b->group == PS_G1) return msm_on_bases<Fp>(ctx, b, 0, d_sc, n, 0, (G1XYZZ*)d_out_xyzz);
  return msm_on_bases<Fp2>(ctx, b, 0, d_sc, n, 0, (G2XYZZ*)d_out_xyzz);
}

}  // namespace ps
}  // extern "C++"

extern "C++" {
namespace {
// out[first .. first + cnt) of the base set's first table = scalars[i] * generator
template <class F>
int fill_from_scalars(ps_ctx* ctx, ps_bases* b, size_t first, const Fr* d_scalars, size_t cnt) {
  if (!cnt) return PS_OK;
  return GroupOps<F>::from_scalars(ctx, (const uint32_t*)d_scalars, cnt, (Affine<F>*)b->tab + first);
}
template <class F>
int export_range(ps_ctx* ctx, const ps_bases* b, size_t first, size_t count, int format, uint8_t* out) {
  if (!out || !count) return PS_OK;
  size_t per = point_bytes(b->group, format);
  uint8_t* d_bytes = ctx->arena.take<uint8_t>(count * per);
  if (!d_bytes) return PS_ERR_ALLOC;
  PS_TRY(GroupOps<F>::encode_affine(ctx, (const Affine<F>*)b->tab + first, count, format, d_bytes));
  return dev_d2h(out, d_bytes, count * per, ctx->stream);
}
// a few points scalar[i] * generator straight to host bytes (verification-key elements)
template <class F>
int export_multiples(ps_ctx* ctx, const Fr* d_scalars, size_t count, int format, uint8_t* out) {
  if (!out || !count) return PS_OK;
  Affine<F>* pts = ctx->arena.take<Affine<F>>(count);
  size_t per = point_bytes(PointBytes<F>::GROUP, format);
  uint8_t* d_bytes = ctx->arena.take<uint8_t>(count * per);
  if (!pts || !d_bytes) return PS_ERR_ALLOC;
  PS_TRY(GroupOps<F>::from_scalars(ctx, (const uint32_t*)d_scalars, count, pts));
  PS_TRY(GroupOps<F>::encode_affine(ctx, (const Affine<F>*)pts, count, format, d_bytes));
  return dev_d2h(out, d_bytes, count * per, ctx->stream);
}
}  // namespace
}  // extern "C++"

// NewGroth16TrustedSetup (groth16.go:64-101) on the device.  A = [Xi | Delta | Alpha], B = [Xi2 | Delta2 | Beta2],
// C = [NioLP | XiT | Xi | Alpha Beta Delta] are filled by the fixed-base kernel from the exponents of setup.cuh.
int ps_g16_setup(ps_ctx* ctx, const ps_qap* qap, const uint8_t* toxic_be, ps_g16_key** key, uint8_t* out_iolp, uint8_t* out_gamma) {
  if (!ctx || !qap || !toxic_be || !key || qap->n < 2) return PS_ERR_ARG;
  PS_TRY(begin_call(ctx));
  const size_t n = qap->n, m = qap->m, nio = qap->n_io, diff = m - nio;
  G16SetupScalars sc;
  PS_TRY(g16_setup_scalars(ctx, qap, toxic_be, &sc));
  ps_g16_key* k = new (std::nothrow) ps_g16_key();
  if (!k) return PS_ERR_ALLOC;
  k->n = n; k->n_nio = nio;
  const Fr *alpha = sc.consts, *beta = sc.consts + 1, *delta = sc.consts + 2, *gamma = sc.consts + 3;
  int rc = g16_key_alloc(k, n + 2, n + 2, nio + (n - 1) + n + 3, batch_window(ctx, 3 * n + nio + 4, 2), batch_window(ctx, n + 2, 1));
  if (rc == PS_OK) rc = fill_from_scalars<Fp>(ctx, k->A, 0, sc.pw, n);
  if (rc == PS_OK) rc = fill_from_scalars<Fp>(ctx, k->A, n, delta, 1);
  if (rc == PS_OK) rc = fill_from_scalars<Fp>(ctx, k->A, n + 1, alpha, 1);
  if (rc == PS_OK) rc = fill_from_scalars<Fp2>(ctx, k->B, 0, sc.pw, n);
  if (rc == PS_OK) rc = fill_from_scalars<Fp2>(ctx, k->B, n, delta, 1);
  if (rc == PS_OK) rc = fill_from_scalars<Fp2>(ctx, k->B, n + 1, beta, 1);
  if (rc == PS_OK) rc = fill_from_scalars<Fp>(ctx, k->C, 0, sc.lp + diff, nio);
  if (rc == PS_OK) rc = fill_from_scalars<Fp>(ctx, k->C, nio, sc.pwt, n - 1);
  if (rc == PS_OK) rc = fill_from_scalars<Fp>(ctx, k->C, nio + (n - 1), sc.pw, n);
  if (rc == PS_OK) rc = fill_from_scalars<Fp>(ctx, k->C, nio + (n - 1) + n, alpha, 3);     // alpha, beta, delta are consecutive
  if (rc == PS_OK) rc = GroupOps<Fp>::tables_finish(ctx, (G1Affine*)k->A->tab, k->A->n, k->A->c, k->A->T);
  if (rc == PS_OK) rc = GroupOps<Fp2>::tables_finish(ctx, (G2Affine*)k->B->tab, k->B->n, k->B->c, k->B->T);
  if (rc == PS_OK) rc = GroupOps<Fp>::tables_finish(ctx, (G1Affine*)k->C->tab, k->C->n, k->C->c, k->C->T);
  // verifier side: IoLP (the first m - n_io variables, divided by gamma) and Gamma in G2, compressed
  if (rc == PS_OK) rc = export_multiples<Fp>(ctx, sc.lp, out_iolp ? diff : 0, PS_FMT_COMPRESSED, out_iolp);
  if (rc == PS_OK) rc = export_multiples<Fp2>(ctx, gamma, out_gamma ? 1 : 0, PS_FMT_COMPRESSED, out_gamma);
  if (rc == PS_OK) rc = dev_sync(ctx->stream);
  if (rc != PS_OK) { ps_g16_key_free(k); return rc; }
  *key = k;
  return PS_OK;
}

// the key's elements back as wire bytes (any output may be NULL): what the Go shim stores into Groth16Setup's fields
int ps_g16_key_export(ps_ctx* ctx, const ps_g16_key* key, int format, uint8_t* xi, uint8_t* xi2, uint8_t* xit, uint8_t* niolp,
                      uint8_t* alpha, uint8_t* beta, uint8_t* delta, uint8_t* beta2, uint8_t* delta2) {
  if (!ctx || !key || (format != PS_FMT_COMPRESSED && format != PS_FMT_AFFINE)) return PS_ERR_ARG;
  PS_TRY(begin_call(ctx));
  const size_t n = key->n, nio = key->n_nio;
  if (key->A->n != n + 2 || key->C->n != nio + (n - 1) + n + 3) return PS_ERR_ARG;   // a per-device slice of a sharded key
  PS_TRY(export_range<Fp>(ctx, key->A, 0, n, format, xi));
  PS_TRY(export_range<Fp>(ctx, key->A, n, 1, format, delta));
  PS_TRY(export_range<Fp>(ctx, key->A, n + 1, 1, format, alpha));
  PS_TRY(export_range<Fp2>(ctx, key->B, 0, n, format, xi2));
  PS_TRY(export_range<Fp2>(ctx, key->B, n, 1, format, delta2));
  PS_TRY(export_range<Fp2>(ctx, key->B, n + 1, 1, format, beta2));
  PS_TRY(export_range<Fp>(ctx, key->C, 0, nio, format, niolp));
  PS_TRY(export_range<Fp>(ctx, key->C, nio, n - 1, format, xit));
  PS_TRY(export_range<Fp>(ctx, key->C, nio + (n - 1) + n + 1, 1, format, beta));
  return dev_sync(ctx->stream);
}

size_t ps_g16_scalar_count(const ps_g16_key* key, int which) {
  if (!key) return 0;
  const ps_bases* b = which == 0 ? key->A : (which == 1 ? key->C : (which == 2 ? key->B : nullptr));
  return b ? b->n : 0;
}

const ps_bases* ps_g16_key_bases(const ps_g16_key* key, int which) {
  if (!key) return nullptr;
  return which == 0 ? key->A : (which == 1 ? key->C : (which == 2 ? key->B : nullptr));
}

int ps_g16_msm_partials(ps_ctx* ctx, const ps_g16_key* key, const void* d_scA, const void* d_scC, const void* d_scB,
                        const size_t first[3], const size_t count[3], void* d_partials) {
  if (!ctx || !key || !d_scA || !d_scC || !d_scB || !first || !count || !d_partials) return PS_ERR_ARG;
  PS_TRY(begin_call(ctx));
  uint8_t* out = (uint8_t*)d_partials;  // [A: 192 B | C: 192 B | B: 384 B]
  PS_TRY(ctx_fork(ctx));
  ForkGuard fg(ctx);
  {
    SecondaryScope scope(ctx);
    PS_TRY(msm_on_bases<Fp2>(ctx, key->B, first[2], (const uint32_t*)d_scB, count[2], 0, (G2XYZZ*)(out + 384)));
  }
  const SegSpec g1segs[2] = {{key->A, first[0], (const uint32_t*)d_scA, count[0], 0, 0},
                             {key->C, first[1], (const uint32_t*)d_scC, count[1], 0, 1}};
  PS_TRY(msm_batch<Fp>(ctx, g1segs, 2, 2, (G1XYZZ*)out));
  return fg.join();
}

int ps_host_alloc(size_t bytes, void** out) {
  if (!out) return PS_ERR_ARG;
#if PS_GPU
  PS_CUDA_TRY(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable));
#else
  *out = malloc(bytes ? bytes : 1);
  if (!*out) return PS_ERR_ALLOC;
#endif
  return PS_OK;
}

void ps_host_free(void* p) {
  if (!p) return;
#if PS_GPU
  cudaFreeHost(p);
#else
  free(p);
#endif
}

int ps_g16_combine(ps_ctx* ctx, const void* d_records, size_t count, size_t stride, uint8_t* outA, uint8_t* outB, uint8_t* outC) {
  if (!ctx || !d_records || !count || !outA || !outB || !outC || stride < 960 || (stride & 15)) return PS_ERR_ARG;
  PS_TRY(begin_call(ctx));
  const uint8_t* recs = (const uint8_t*)d_records;
  G1XYZZ* resG1 = ctx->arena.take<G1XYZZ>(2);
  if (!resG1) return PS_ERR_ALLOC;
  PS_TRY(ctx_fork(ctx));
  ForkGuard fg(ctx);
  {
    SecondaryScope scope(ctx);
    G2XYZZ* resG2 = ctx->arena.take<G2XYZZ>(1);
    if (!resG2) return PS_ERR_ALLOC;
    const int o0[2] = {384, 384}, o1[2] = {-1, -1};
    PS_TRY(GroupOps<Fp2>::record_sum(ctx, 1, (uint32_t)count, recs, (uint32_t)stride, o0, o1, resG2));
    PS_TRY(encode_points_staged<Fp2>(ctx, resG2, 1, 96));
  }
  const int o0[2] = {0, 192}, o1[2] = {-1, 768};
  PS_TRY(GroupOps<Fp>::record_sum(ctx, 2, (uint32_t)count, recs, (uint32_t)stride, o0, o1, resG1));
  PS_TRY(encode_points_staged<Fp>(ctx, resG1, 2, 0));
  PS_TRY(fg.join());
  PS_TRY(dev_sync(ctx->stream));
  memcpy(outA, ctx->h_stage, 48);
  memcpy(outC, ctx->h_stage + 48, 48);
  memcpy(outB, ctx->h_stage + 96, 96);
  return PS_OK;
}

// ---- PHGR13 -------------------------------------------------------------------------------------------
int ps_phgr13_key_load(ps_ctx* ctx, size_t n_gates, size_t n_mid, int format, const uint8_t* gsi, const uint8_t* vs,
                       const uint8_t* ws, const uint8_t* ys, const uint8_t* vas, const uint8_t* was, const uint8_t* yas,
                       const uint8_t* vbs, const uint8_t* wbs, const uint8_t* ybs, ps_phgr13_key** key) {
  if (!key || !gsi || n_gates < 2) return PS_ERR_ARG;
  if (n_mid && (!vs || !ws || !ys || !vas || !was || !yas || !vbs || !wbs || !ybs)) return PS_ERR_ARG;
  if (format != PS_FMT_COMPRESSED && format != PS_FMT_AFFINE) return PS_ERR_ARG;
  PS_TRY(begin_call(ctx));
  ps_phgr13_key* k = new (std::nothrow) ps_phgr13_key();
  if (!k) return PS_ERR_ALLOC;
  k->n = n_gates; k->n_mid = n_mid;
  const uint8_t* singles[6] = {gsi, vs, ys, vas, was, yas};
  const size_t counts[6] = {n_gates - 1, n_mid, n_mid, n_mid, n_mid, n_mid};
  int rc = phgr13_key_alloc(ctx, k, n_gates, n_mid);
  for (int i = 0; i < 6 && rc == PS_OK; i++) {
    rc = bases_concat_into<Fp>(ctx, k->g1[i], format, &singles[i], &counts[i], 1);
    if (rc == PS_OK) rc = ctx->arena.reset();
  }
  const uint8_t* zs[3] = {vbs, wbs, ybs};
  const size_t zc[3] = {n_mid, n_mid, n_mid};
  if (rc == PS_OK) rc = bases_concat_into<Fp>(ctx, k->g1[6], format, zs, zc, 3);
  if (rc == PS_OK) rc = ctx->arena.reset();
  if (rc == PS_OK) rc = bases_concat_into<Fp2>(ctx, k->ws, format, &ws, &n_mid, 1);
  if (rc != PS_OK) { ps_phgr13_key_free(k); return rc; }
  *key = k;
  return PS_OK;
}

// NewPHGR13TrustedSetup (pinochio.go:93-176) on the device: the resident evaluation key and, on request, the
// verification key as compressed bytes:
//   out_vk_fixed (7 elements): av (G2 96 B) | aw (G1 48) | ay (G2 96) | gamma (G2 96) | bgamma (G1 48) | bgamma2 (G2 96) | yts (G2 96)
//   out_vk_vs / out_vk_ws / out_vk_ys: the commitments of ALL n_vars variables (48 / 96 / 48 B each)
int ps_phgr13_setup(ps_ctx* ctx, const ps_qap* qap, const uint8_t* toxic_be, ps_phgr13_key** key, uint8_t* out_vk_fixed,
                    uint8_t* out_vk_vs, uint8_t* out_vk_ws, uint8_t* out_vk_ys) {
  if (!ctx || !qap || !toxic_be || !key || qap->n < 2) return PS_ERR_ARG;
  PS_TRY(begin_call(ctx));
  const size_t n = qap->n, m = qap->m, nmid = qap->n_io, diff = m - nmid;
  Phgr13SetupScalars sc;
  PS_TRY(phgr13_setup_scalars(ctx, qap, toxic_be, &sc));
  ps_phgr13_key* k = new (std::nothrow) ps_phgr13_key();
  if (!k) return PS_ERR_ALLOC;
  k->n = n; k->n_mid = nmid;
  // g1[]: gsi vs ys vas was yas [vbs|wbs|ybs];  ek[]: vs ws ys vas was yas vbs wbs ybs
  const int ek_of_g1[6] = {-1, 0, 2, 3, 4, 5};
  int rc = phgr13_key_alloc(ctx, k, n, nmid);
  if (rc == PS_OK) rc = fill_from_scalars<Fp>(ctx, k->g1[0], 0, sc.pw, n - 1);
  for (int i = 1; i < 6 && rc == PS_OK; i++) rc = fill_from_scalars<Fp>(ctx, k->g1[i], 0, sc.ek[ek_of_g1[i]] + diff, nmid);
  for (int t = 0; t < 3 && rc == PS_OK; t++) rc = fill_from_scalars<Fp>(ctx, k->g1[6], (size_t)t * nmid, sc.ek[6 + t] + diff, nmid);
  if (rc == PS_OK) rc = fill_from_scalars<Fp2>(ctx, k->ws, 0, sc.ek[1] + diff, nmid);
  for (int i = 0; i < 7 && rc == PS_OK; i++) rc = GroupOps<Fp>::tables_finish(ctx, (G1Affine*)k->g1[i]->tab, k->g1[i]->n, k->g1[i]->c, k->g1[i]->T);
  if (rc == PS_OK) rc = GroupOps<Fp2>::tables_finish(ctx, (G2Affine*)k->ws->tab, k->ws->n, k->ws->c, k->ws->T);
  if (rc == PS_OK && out_vk_fixed) {
    const Fr* cs = sc.consts;   // av aw ay gamma bgamma t(s)*ry
    uint8_t* o = out_vk_fixed;
    rc = export_multiples<Fp2>(ctx, cs + 0, 1, PS_FMT_COMPRESSED, o);
    if (rc == PS_OK) rc = export_multiples<Fp>(ctx, cs + 1, 1, PS_FMT_COMPRESSED, o + 96);
    if (rc == PS_OK) rc = export_multiples<Fp2>(ctx, cs + 2, 1, PS_FMT_COMPRESSED, o + 144);
    if (rc == PS_OK) rc = export_multiples<Fp2>(ctx, cs + 3, 1, PS_FMT_COMPRESSED, o + 240);
    if (rc == PS_OK) rc = export_multiples<Fp>(ctx, cs + 4, 1, PS_FMT_COMPRESSED, o + 336);
    if (rc == PS_OK) rc = export_multiples<Fp2>(ctx, cs + 4, 1, PS_FMT_COMPRESSED, o + 384);
    if (rc == PS_OK) rc = export_multiples<Fp2>(ctx, cs + 5, 1, PS_FMT_COMPRESSED, o + 480);
  }
  if (rc == PS_OK) rc = export_multiples<Fp>(ctx, sc.ek[0], out_vk_vs ? m : 0, PS_FMT_COMPRESSED, out_vk_vs);
  if (rc == PS_OK) rc = export_multiples<Fp2>(ctx, sc.ek[1], out_vk_ws ? m : 0, PS_FMT_COMPRESSED, out_vk_ws);
  if (rc == PS_OK) rc = export_multiples<Fp>(ctx, sc.ek[2], out_vk_ys ? m : 0, PS_FMT_COMPRESSED, out_vk_ys);
  if (rc == PS_OK) rc = dev_sync(ctx->stream);
  if (rc != PS_OK) { ps_phgr13_key_free(k); return rc; }
  *key = k;
  return PS_OK;
}

// the evaluation key back as wire bytes (any output may be NULL), the order of ps_phgr13_key_load's arguments
int ps_phgr13_key_export(ps_ctx* ctx, const ps_phgr13_key* key, int format, uint8_t* gsi, uint8_t* vs, uint8_t* ws, uint8_t* ys,
                         uint8_t* vas, uint8_t* was, uint8_t* yas, uint8_t* vbs, uint8_t* wbs, uint8_t* ybs) {
  if (!ctx || !key || (format != PS_FMT_COMPRESSED && format != PS_FMT_AFFINE)) return PS_ERR_ARG;
  PS_TRY(begin_call(ctx));
  const size_t nm = key->n_mid;
  uint8_t* singles[6] = {gsi, vs, ys, vas, was, yas};
  for (int i = 0; i < 6; i++) PS_TRY(export_range<Fp>(ctx, key->g1[i], 0, key->g1[i]->n, format, singles[i]));
  uint8_t* zs[3] = {vbs, wbs, ybs};
  for (int t = 0; t < 3; t++) PS_TRY(export_range<Fp>(ctx, key->g1[6], (size_t)t * nm, nm, format, zs[t]));
  PS_TRY(export_range<Fp2>(ctx, key->ws, 0, nm, format, ws));
  return dev_sync(ctx->stream);
}

void ps_phgr13_key_free(ps_phgr13_key* key) {
  if (!key) return;
  for (auto* b : key->g1) ps_bases_free(b);
  ps_bases_free(key->ws);
  dev_free(key->slab_g1);
  delete key;
}

int ps_phgr13_prove(ps_ctx* ctx, const ps_phgr13_key* key, const ps_qap* qap, const uint8_t* witness_be, uint8_t* out432,
                    uint8_t* out_h) {
  if (!key || !qap || !witness_be || !out432) return PS_ERR_ARG;
  if (key->n != qap->n || key->n_mid != qap->n_io) return PS_ERR_LENGTH;
  PS_TRY(begin_call(ctx));
  const size_t n = qap->n, nmid = qap->n_io, diff = qap->m - qap->n_io;
  QuotientBufs qb;
  PS_TRY(run_quotient(ctx, qap, witness_be, &qb));
  G1XYZZ* resG1 = ctx->arena.take<G1XYZZ>(7);
  G2XYZZ* resG2 = ctx->arena.take<G2XYZZ>(1);
  if (!resG1 || !resG2) return PS_ERR_ALLOC;
  const uint32_t* wmid = (const uint32_t*)(qb.w + diff);
  // wss (G2) is independent of the seven G1 sums: second stream, like Groth16's B
  PS_TRY(ctx_fork(ctx));
  ForkGuard fg(ctx);
  {
    SecondaryScope scope(ctx);
    PS_TRY(msm_on_bases<Fp2>(ctx, key->ws, 0, wmid, nmid, 1, resG2));               // wss
    PS_TRY(encode_points_staged<Fp2>(ctx, resG2, 1, 7 * 48));
  }
  // hs, vss, yss, vass, wass, yass and gz = <w, vbs> + <w, wbs> + <w, ybs> as ONE pipeline: nine segments into
  // seven outputs; the shared scalars solution[diff:] are decomposed per segment, sorted and reduced once
  SegSpec segs[9];
  segs[0] = SegSpec{key->g1[0], 0, (const uint32_t*)qb.h, n - 1, 1, 0};
  for (int i = 1; i < 6; i++) segs[i] = SegSpec{key->g1[i], 0, wmid, nmid, 1, i};
  for (int t = 0; t < 3; t++) segs[6 + t] = SegSpec{key->g1[6], (size_t)t * nmid, wmid, nmid, 1, 6};
  PS_TRY(msm_batch<Fp>(ctx, segs, 9, 7, resG1));
  PS_TRY(encode_points_staged<Fp>(ctx, resG1, 7, 0));
  PS_TRY(fg.join());
  if (out_h) PS_TRY(export_fr(ctx, qb.h, n - 1, out_h));
  PS_TRY(check_err_flag(ctx, qb.enc_err, PS_ERR_ENCODING));
  PS_TRY(check_err_flag(ctx, qb.flag, PS_ERR_REMAINDER));
  memcpy(out432, ctx->h_stage, 432);
  return PS_OK;
}

// ---- measurement ----------------------------------------------------------------------------------------
int ps_bench_intpipe(ps_ctx* ctx, int variant, int iters, double* inst_per_s, double* ms_out) {
  if (!ctx || !inst_per_s || variant < 0 || variant > 3 || iters < 1) return PS_ERR_ARG;
#if PS_GPU
  PS_TRY(begin_call(ctx));
  uint32_t* d_out = ctx->arena.take<uint32_t>(4);
  if (!d_out) return PS_ERR_ALLOC;
  const int blocks = ctx->sm_count * 8, threads = 256;
  cudaEvent_t e0, e1;
  PS_CUDA_TRY(cudaEventCreate(&e0)); PS_CUDA_TRY(cudaEventCreate(&e1));
  for (int rep = 0; rep < 2; rep++) {  // first pass warms up
    PS_CUDA_TRY(cudaEventRecord(e0, ctx->stream));
    switch (variant) {
      case 0: k_intpipe<0><<<blocks, threads, 0, ctx->stream>>>(d_out, iters, 12345u); break;
      case 1: k_intpipe<1><<<blocks, threads, 0, ctx->stream>>>(d_out, iters, 12345u); break;
      case 2: k_intpipe<2><<<blocks, threads, 0, ctx->stream>>>(d_out, iters, 12345u); break;
      default: k_intpipe<3><<<blocks, threads, 0, ctx->stream>>>(d_out, iters, 12345u); break;
    }
    PS_CUDA_TRY(cudaEventRecord(e1, ctx->stream));
    PS_CUDA_TRY(cudaEventSynchronize(e1));
    launch_counter()++;
  }
  float ms = 0;
  PS_CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  double inst = (double)blocks * threads * (double)iters * intpipe_inst_per_iter(variant);
  *inst_per_s = inst / (ms * 1e-3);
  if (ms_out) *ms_out = ms;
  return PS_OK;
#else
  (void)ms_out;
  return PS_ERR_UNSUPPORTED;
#endif
}

int ps_bench_fieldmul(ps_ctx* ctx, int field, int iters, double* mul_per_s, double* ms_out) {
  if (!ctx || !mul_per_s || field < 0 || field > 1 || iters < 1) return PS_ERR_ARG;
#if PS_GPU
  PS_TRY(begin_call(ctx));
  const int blocks = ctx->sm_count * 4, threads = 256;
  const size_t nthreads = (size_t)blocks * threads;
  void* d_io = ctx->arena.take<Fp>(2 * nthreads);
  if (!d_io) return PS_ERR_ALLOC;
  PS_TRY(dev_memset(d_io, 0x5a, 2 * nthreads * sizeof(Fp), ctx->stream));
  cudaEvent_t e0, e1;
  PS_CUDA_TRY(cudaEventCreate(&e0)); PS_CUDA_TRY(cudaEventCreate(&e1));
  for (int rep = 0; rep < 2; rep++) {
    PS_CUDA_TRY(cudaEventRecord(e0, ctx->stream));
    if (field == 0) k_fieldmul<Fr><<<blocks, threads, 0, ctx->stream>>>((Fr*)d_io, iters);
    else k_fieldmul<Fp><<<blocks, threads, 0, ctx->stream>>>((Fp*)d_io, iters);
    PS_CUDA_TRY(cudaEventRecord(e1, ctx->stream));
    PS_CUDA_TRY(cudaEventSynchronize(e1));
    launch_counter()++;
  }
  float ms = 0;
  PS_CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  *mul_per_s = (double)nthreads * 2.0 * iters / (ms * 1e-3);
  if (ms_out) *ms_out = ms;
  return PS_OK;
#else
  (void)ms_out;
  return PS_ERR_UNSUPPORTED;
#endif
}

}  // extern "C"
