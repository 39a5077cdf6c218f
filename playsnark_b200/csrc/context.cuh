// The per-GPU context behind the C ABI's opaque ps_ctx handle.
#pragma once
#include "backend.cuh"
#include <utility>

#ifndef PS_BUCKET_COST
#define PS_BUCKET_COST 70   // see msm_pick_window_full (group_ops.cuh)
#endif

namespace ps {
// Twiddle tables for one transform size, resident on the device (built by ntt_tables_build, ntt.cuh).
struct NttTables {
  int log_n = -1;
  Fr* tw = nullptr;      // omega^i, i < max(n/2, 1)
  Fr* tw_inv = nullptr;  // omega^-i
  void release() { dev_free(tw); dev_free(tw_inv); tw = tw_inv = nullptr; log_n = -1; }
};
}  // namespace ps

#ifndef PS_SCATTER_DEFAULT
#define PS_SCATTER_DEFAULT 1
#endif

struct ps_ctx {
  int device = 0;
  ps::ps_stream_t stream = nullptr;
  bool own_stream = false;
  int sm_count = 148;
  ps::Arena arena;                 // per-call scratch, persists across calls
  // secondary stream + scratch: lets an independent MSM (Groth16's G2 one) overlap the others
  ps::ps_stream_t stream2 = nullptr;
  ps::Arena arena2;
  void* ev_fork = nullptr;         // cudaEvent_t: inputs ready on `stream`
  void* ev_join = nullptr;         // cudaEvent_t: secondary work done on `stream2`
  bool timing_events = true;       // phase events are only recorded for work on the primary stream
  ps::NttTables ntt_cache[31];     // twiddles by log2(size), built on first use
  void* fixed_base[2] = {nullptr, nullptr};  // 32 x 255 affine multiples of the G1 / G2 generator
  // phase events of the last MSM (cudaEvent_t): start, sorted, accumulated, combined, reduced
  void* ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  bool ev_valid = false;
  // phase events of the last Groth16 prove: start, quotient done, MSM A, MSM C, MSM B, encoded
  void* evp[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  bool evp_valid = false;
  // phase events of the last ps_g16_verify_batch: start, uploaded, decoded, weighted, io sums, Miller loops, tree, root
  // check, bisection done
  void* evv[9] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  bool evv_valid = false;
  // point decoding rejects points outside the prime-order subgroup (kilic's FromCompressed does); 0 skips the
  // r-multiplication for key material the caller vouches for
  int subgroup_check = 1;
  // lowest levels of the interpolation tree in one shared-memory kernel (interp.cuh); 0 = level by level
  int interp_fused = 1;
  // accumulate grid of small MSMs: 1 = whole waves with the wave count rounded down (longer chunks), 0 = rounded up
  int msm_wave_floor = 1;
  // latency-bound tail kernels of the MSM: 1 = a team of four lanes per group operation (team.cuh), 0 = one thread
  int msm_team = 1;
  // base sets loaded from now on are meant to be summed in this many index ranges (sharded proofs)
  int msm_shards = 1;
  // bucket sort of the MSM entries: 0 = one-pass counting sort, 1 = two-level sort from 2^25 entries (msm.cuh),
  // 2 = two-level sort whenever possible (tests)
  int msm_scatter = PS_SCATTER_DEFAULT;
  // window model: time of one bucket (merge + reduction) in field products, a mixed addition being 10
  int msm_bucket_cost = PS_BUCKET_COST;
  // small page-locked staging area for results: a device-to-host copy into pageable memory would block
  // the host until the producing stream has drained, which serialises work meant for the other stream
  uint8_t* h_stage = nullptr;
  static constexpr size_t H_STAGE_BYTES = 4096;
};

namespace ps {
// twiddle tables by size, built on first use (defined in capi_poly.cu, the translation unit of the Fr kernels)
int ctx_ntt_tables(ps_ctx* ctx, int log_n, const NttTables** out);
inline int ctx_event(ps_ctx* ctx, int i) {
  if (!ctx->timing_events) return PS_OK;
#if PS_GPU
  if (ctx->ev[i]) PS_CUDA_TRY(cudaEventRecord((cudaEvent_t)ctx->ev[i], ctx->stream));
#else
  (void)ctx; (void)i;
#endif
  return PS_OK;
}
inline int ctx_verify_event(ps_ctx* ctx, int i) {
#if PS_GPU
  if (ctx->evv[i]) PS_CUDA_TRY(cudaEventRecord((cudaEvent_t)ctx->evv[i], ctx->stream));
#else
  (void)ctx; (void)i;
#endif
  return PS_OK;
}
inline int ctx_prove_event(ps_ctx* ctx, int i) {
#if PS_GPU
  if (ctx->evp[i]) PS_CUDA_TRY(cudaEventRecord((cudaEvent_t)ctx->evp[i], ctx->stream));
#else
  (void)ctx; (void)i;
#endif
  return PS_OK;
}

// Runs the enclosed calls on the context's secondary stream / arena (host code is sequential, so
// swapping the two fields is enough); the destructor swaps back.
struct SecondaryScope {
  ps_ctx* ctx;
  explicit SecondaryScope(ps_ctx* c) : ctx(c) { swap(); ctx->timing_events = false; }
  ~SecondaryScope() { swap(); ctx->timing_events = true; }
  void swap() {
    ps_stream_t s = ctx->stream; ctx->stream = ctx->stream2; ctx->stream2 = s;
    std::swap(ctx->arena.blocks, ctx->arena2.blocks);
    std::swap(ctx->arena.stream, ctx->arena2.stream);
  }
};
// secondary stream waits for everything enqueued so far on the primary one
inline int ctx_fork(ps_ctx* ctx) {
#if PS_GPU
  PS_CUDA_TRY(cudaEventRecord((cudaEvent_t)ctx->ev_fork, ctx->stream));
  PS_CUDA_TRY(cudaStreamWaitEvent(ctx->stream2, (cudaEvent_t)ctx->ev_fork, 0));
#else
  (void)ctx;
#endif
  return PS_OK;
}
// primary stream waits for everything enqueued so far on the secondary one
inline int ctx_join(ps_ctx* ctx) {
#if PS_GPU
  PS_CUDA_TRY(cudaEventRecord((cudaEvent_t)ctx->ev_join, ctx->stream2));
  PS_CUDA_TRY(cudaStreamWaitEvent(ctx->stream, (cudaEvent_t)ctx->ev_join, 0));
#else
  (void)ctx;
#endif
  return PS_OK;
}
}  // namespace ps
