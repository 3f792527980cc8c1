// integrate.cu — TSDF integration of point clouds into the block-hashed layer: the job driver and
// the C ABI of the integrator.
//
// Replaces voxblox::TsdfIntegratorBase::integratePointCloud (Simple / Merged semantics, R1-R6 of
// SURVEY.md §8a); reference call site coxgraph/include/coxgraph/map_comm/tsdf_recover.h:75.
//
// One job = one frame, or a batch of frames fused into the same layer (the loop of
// tsdf_recover.h:71-86).  All frames of a job go through every stage together (DESIGN.md §4):
//  front half (integrate_front.cu) — points to one ray per bundle (R1, R2, R6)
//  back half (integrate_back.cu)   — rays to voxels (R3, R4, R5)
// A job too large for one pass runs as several groups of frames, each through both halves.
// Per-voxel order is (frame, non-clearing before clearing, bundle key ascending) — the oracle's
// canonical order — independent of scheduling.
#include <string.h>

#include <algorithm>
#include <vector>

#include "host_stage.cuh"
#include "integrate.cuh"

namespace cg {

// Device-side fill used instead of cudaMemsetAsync on the compute stream: a memset may be
// executed by a copy engine, where it would queue behind the (large) host->device transfers of
// the pipelined batch path and stall the kernels that follow it.
__global__ void k_fill_words(uint32_t* __restrict__ p, uint32_t v, size_t n) {
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x)
    p[i] = v;
}
cudaError_t fill_bytes(void* p, int byte, size_t bytes, cudaStream_t s) {
  const size_t n = bytes / 4;
  if (n == 0) return cudaSuccess;
  const uint32_t v = 0x01010101u * static_cast<uint32_t>(byte & 0xFF);
  const unsigned grid = static_cast<unsigned>(std::min<size_t>((n + 255) / 256, 148 * 8));
  k_fill_words<<<grid, 256, 0, s>>>(static_cast<uint32_t*>(p), v, n);
  return cudaGetLastError();
}

// ------------------------------------------------------------------ host orchestration
static IntegratorParams make_params(const cg_layer* L, const cg_integrator_config* c, int freespace) {
  IntegratorParams P;
  P.trunc = c->default_truncation_distance;
  P.max_weight = c->max_weight;
  P.min_ray = c->min_ray_length_m;
  P.max_ray = c->max_ray_length_m;
  P.voxel_size = L->v.voxel_size;
  P.voxel_size_inv = L->v.voxel_size_inv;
  P.sparsity_factor = c->sparsity_compensation_factor;
  P.carving = c->voxel_carving_enabled;
  P.const_weight = c->use_const_weight;
  P.allow_clear = c->allow_clear;
  P.weight_dropoff = c->use_weight_dropoff;
  P.use_sparsity = c->use_sparsity_compensation_factor;
  P.order_mode = c->integration_order_mode;
  P.freespace = freespace;
  // anti-grazing belongs to the merged integrator only (the simple one never looks at it)
  P.anti_grazing = (c->enable_anti_grazing && c->method == CG_METHOD_MERGED) ? 1 : 0;
  return P;
}

// CG_OK when the integrator can run `cfg`; `report`: also set the error text
static int32_t check_config(const cg_integrator_config* cfg, bool report) {
  if (cfg->method == CG_METHOD_FAST) {
    if (report)
      set_error("method FAST is order- and wall-clock-dependent in the reference and has no "
                "deterministic device form; use MERGED or SIMPLE");
    return CG_ERR_UNSUPPORTED;
  }
  if (cfg->method != CG_METHOD_MERGED && cfg->method != CG_METHOD_SIMPLE) return CG_ERR_INVALID_ARG;
  if (!(cfg->default_truncation_distance > 0.0f) || !(cfg->max_ray_length_m > 0.0f)) {
    if (report) set_error("invalid integrator config");
    return CG_ERR_INVALID_ARG;
  }
  return CG_OK;
}

static int32_t check_offsets(const uint64_t* offs, size_t F) {
  for (size_t f = 0; f < F; ++f)
    if (offs[f + 1] < offs[f]) {
      set_error("frame_offsets must be non-decreasing");
      return CG_ERR_INVALID_ARG;
    }
  return CG_OK;
}

// points of one group at most: a job with more runs as several groups of whole frames
static size_t max_group_points() {
  return env_size("CG_MAX_GROUP_POINTS", size_t(48) << 20);
}

// Back half of a front half the host has synchronised on and digested.
static int32_t integrate_rays(cg_layer* L, const FrontBufs& fb, const IntegratorParams& P,
                              cg_integrate_stats* stats) {
  const uint32_t num_rays = static_cast<uint32_t>(fb.h_counters->rays);
  const size_t num_pairs = fb.h_counters->pairs;
  if (stats) stats->points_beyond_reach += fb.h_counters->far_dropped;
  if (num_rays == 0 || num_pairs == 0) return CG_OK;
  if (stats) {
    stats->rays += num_rays;
    stats->voxel_updates += num_pairs;
  }
  return run_back_half(L->ctx, fb, L, P, num_rays, num_pairs, fb.h_counters->segments, stats);
}

// frames [f0, f1) of the job as one group; splits itself when the pair list would not fit
static int32_t integrate_group(cg_layer* L, const cg_integrator_config* cfg,
                               const IntegratorParams& P, const float* h_poses,
                               const float* d_points, const uint8_t* d_colors,
                               const uint64_t* offs, size_t f0, size_t f1,
                               cg_integrate_stats* stats, int attempt = 0) {
  cg_context* ctx = L->ctx;
  cudaStream_t s = ctx->stream;
  const size_t F = f1 - f0;
  const size_t total = offs[f1] - offs[f0];  // points of the group = upper bound on rays
  if (total == 0) return CG_OK;
  if (total > 0x7FFFFFF0ull || F > (1u << 20)) {
    set_error("too many points / frames in one group");
    return CG_ERR_INVALID_ARG;
  }
  auto halves = [&]() -> int32_t {
    const size_t mid = f0 + F / 2;
    int32_t rc = integrate_group(L, cfg, P, h_poses, d_points, d_colors, offs, f0, mid, stats);
    if (rc) return rc;
    return integrate_group(L, cfg, P, h_poses, d_points, d_colors, offs, mid, f1, stats);
  };
  bool need_split = false;
  int32_t rc = front_enqueue(ctx, *ctx, s, L->v.err, L, cfg, P, d_points, d_colors, offs, f0, f1,
                             attempt, &need_split);
  if (rc) return rc;
  if (need_split) return halves();
  CG_CUDA(cudaStreamSynchronize(s));
  CG_CUDA(cudaGetLastError());
  switch (front_digest(ctx, *ctx, cfg->method == CG_METHOD_MERGED, F, attempt, &rc)) {
    case kFrontRetry:
      return integrate_group(L, cfg, P, h_poses, d_points, d_colors, offs, f0, f1, stats, attempt + 1);
    case kFrontSplit:
      return halves();
    case kFrontFail:
      return rc;
    case kFrontOk:
      break;
  }
  return integrate_rays(L, *ctx, P, stats);
}

// One job.  `queued`: the front half of the whole job, queued by cg_prepare_batch_* into a set of
// its own and completed by `queued_done` (h_poses / offs are then that job's copies).  It is used
// when it came out right; otherwise — a point outside the key box, too many voxel visits for one
// group, a ray out of range — it is dropped and the job runs the plain way, which regroups,
// retries and reports.  `inputs_ready`: the staged copy of d_points / d_colors, which the plain way
// must wait for (a queued front half already did).
static int32_t integrate_job(cg_layer* L, const cg_integrator_config* cfg, size_t F,
                             const float* h_poses, const float* d_points, const uint8_t* d_colors,
                             const uint64_t* offs, int freespace, cg_integrate_stats* stats,
                             const FrontBufs* queued = nullptr, cudaEvent_t queued_done = nullptr,
                             cudaEvent_t inputs_ready = nullptr) {
  if (!L || !cfg || !h_poses || !offs || (offs[F] > offs[0] && (!d_points || !d_colors))) {
    set_error("cg_integrate: null argument");
    return CG_ERR_INVALID_ARG;
  }
  int32_t rc = check_offsets(offs, F);
  if (!rc) rc = check_config(cfg, true);
  if (rc) return rc;
  cg_context* ctx = L->ctx;
  CG_CUDA(cudaSetDevice(ctx->device));
  const IntegratorParams P = make_params(L, cfg, freespace);
  const int64_t blocks_before = L->num_blocks;
  if (stats) {
    memset(stats, 0, sizeof(*stats));
    stats->points_in = offs[F] - offs[0];
  }
  bool done = false;
  if (queued) {
    CG_CUDA(cudaEventSynchronize(queued_done));
    int32_t digest_rc = CG_OK;  // (attempt 3: a point outside the key box is not retried here)
    if (front_digest(ctx, *queued, cfg->method == CG_METHOD_MERGED, F, 3, &digest_rc) == kFrontOk &&
        !(queued->h_counters->err & kErrOutOfRange)) {
      rc = integrate_rays(L, *queued, P, stats);
      done = true;
    }
  }
  if (!done) {
    if (inputs_ready) CG_CUDA(cudaStreamWaitEvent(ctx->stream, inputs_ready, 0));
    // poses and frame offsets (relative to the job's first point) go up once per job
    rc = upload_frame_tables(*ctx, F, h_poses, offs, ctx->stream);
    if (rc) return rc;
    const size_t group_points = max_group_points();
    size_t f0 = 0;
    while (f0 < F && rc == CG_OK) {
      size_t f1 = f0 + 1;
      while (f1 < F && offs[f1 + 1] - offs[f0] <= group_points) ++f1;
      rc = integrate_group(L, cfg, P, h_poses, d_points, d_colors, offs, f0, f1, stats);
      f0 = f1;
    }
  }
  const int32_t rc2 = finish_call(L, nullptr);
  if (stats) stats->blocks_allocated = L->num_blocks - blocks_before;
  return rc ? rc : rc2;
}

static int32_t stage_inputs(cg_context* ctx, const float* pts, const uint8_t* cols, size_t n) {
  CG_CUDA(cudaSetDevice(ctx->device));
  CG_CUDA(ctx->points.reserve(n * 3 * sizeof(float)));
  CG_CUDA(ctx->colors.reserve(n * 4));
  StageScope sc(ctx, kStageTransfer, 0);
  // pageable inputs (std::vector clouds of the drop-in call) go through worker threads and a
  // pinned bounce buffer (host_stage.cu); CG_STAGE_THREADS=0 restores the plain copies
  static const int threads = static_cast<int>(env_size("CG_STAGE_THREADS", 3));
  CG_CUDA(stage_begin(ctx->stager, ctx->stream));
  CG_CUDA(stage_to_device(&ctx->stager, ctx->points.p, pts, n * 3 * sizeof(float), ctx->stream,
                          threads));
  CG_CUDA(stage_to_device(&ctx->stager, ctx->colors.p, cols, n * 4, ctx->stream, threads));
  return CG_OK;
}

// The points cg_stage_batch_async staged in `slot` and the event that completes their copy;
// `offs` must cover exactly those points.  `who` names the entry point in the error text.
struct StagedInputs {
  const float* pts;
  const uint8_t* cols;
  cudaEvent_t ready;
};
static int32_t staged_inputs(const char* who, cg_layer* L, const cg_integrator_config* cfg,
                             const float* poses, int32_t slot, size_t F, const uint64_t* offs,
                             StagedInputs* in) {
  if (!L || !cfg || !poses || !offs || slot < 0 || slot > 1 || !L->ctx->stage_ready[slot]) {
    set_error("%s: invalid argument (nothing staged in this slot?)", who);
    return CG_ERR_INVALID_ARG;
  }
  cg_context* ctx = L->ctx;
  if (offs[0] != 0 || offs[F] != ctx->stage_points[slot]) {
    set_error("%s: frame_offsets must cover exactly the %zu staged points", who,
              ctx->stage_points[slot]);
    return CG_ERR_INVALID_ARG;
  }
  *in = StagedInputs{ctx->stage_pts[slot].as<float>(), ctx->stage_cols[slot].as<uint8_t>(),
                     ctx->stage_ready[slot]};
  return CG_OK;
}

// ---- pipelined jobs: the front half of a later job beside the back half of the current one
static int32_t prepare_job(cg_layer* L, const cg_integrator_config* cfg, size_t F,
                           const float* poses, const float* d_pts, const uint8_t* d_cols,
                           const uint64_t* offs, int32_t freespace, int32_t slot,
                           cudaEvent_t inputs_ready) {
  if (!L || !cfg || !poses || !offs || slot < 0 || slot > 1) {
    set_error("cg_prepare_batch: invalid argument");
    return CG_ERR_INVALID_ARG;
  }
  int32_t rc = check_offsets(offs, F);
  if (rc) return rc;
  cg_context* ctx = L->ctx;
  CG_CUDA(cudaSetDevice(ctx->device));
  FrontBufs& fb = ctx->prep[slot];
  if (!ctx->prep_stream) CG_CUDA(cudaStreamCreateWithFlags(&ctx->prep_stream, cudaStreamNonBlocking));
  if (!ctx->prep_done[slot]) {
    CG_CUDA(cudaEventCreateWithFlags(&ctx->prep_done[slot], cudaEventDisableTiming));
    CG_CUDA(init_front_words(fb));
  }
  cg_context::PreparedJob& pj = ctx->prepared[slot];
  pj.valid = true;
  pj.front_queued = false;
  pj.cfg = *cfg;
  pj.poses.assign(poses, poses + 7 * F);
  pj.offs.resize(F + 1);
  for (size_t f = 0; f <= F; ++f) pj.offs[f] = offs[f] - offs[0];
  pj.d_points = d_pts ? d_pts + 3 * offs[0] : nullptr;
  pj.d_colors = d_cols ? d_cols + 4 * offs[0] : nullptr;
  pj.freespace = freespace;
  pj.voxel_size = L->v.voxel_size;
  pj.inputs_ready = inputs_ready;
  const size_t total = pj.offs[F];
  // the fast path: a valid merged / simple job that is one group; everything else is left to the
  // plain path inside cg_integrate_prepared (which also reports the errors)
  if (check_config(cfg, false) != CG_OK || total == 0 || total > max_group_points() ||
      total > 0x7FFFFFF0ull || F > (1u << 20) || !d_pts || !d_cols)
    return CG_OK;
  const IntegratorParams P = make_params(L, cfg, freespace);
  cudaStream_t ps = ctx->prep_stream;
  // the inputs were produced on the context's stream (or by the staged copy): order behind them
  if (!ctx->wait_event) CG_CUDA(cudaEventCreateWithFlags(&ctx->wait_event, cudaEventDisableTiming));
  CG_CUDA(cudaEventRecord(ctx->wait_event, ctx->stream));
  CG_CUDA(cudaStreamWaitEvent(ps, ctx->wait_event, 0));
  if (inputs_ready) CG_CUDA(cudaStreamWaitEvent(ps, inputs_ready, 0));
  CG_CUDA(fill_bytes(fb.d_front_err, 0, sizeof(int32_t), ps));
  rc = upload_frame_tables(fb, F, pj.poses.data(), pj.offs.data(), ps);
  if (rc) return rc;
  bool need_split = false;
  rc = front_enqueue(ctx, fb, ps, fb.d_front_err, L, cfg, P, pj.d_points, pj.d_colors,
                     pj.offs.data(), 0, F, 0, &need_split);
  if (rc) return rc;
  if (need_split) {  // does not fit one group: drain and leave the job to the plain path
    CG_CUDA(cudaStreamSynchronize(ps));
    return CG_OK;
  }
  CG_CUDA(cudaEventRecord(ctx->prep_done[slot], ps));
  pj.front_queued = true;
  return CG_OK;
}

}  // namespace cg

using namespace cg;

extern "C" {

int32_t cg_prepare_batch_device(cg_layer* L, const cg_integrator_config* cfg, size_t F,
                                const float* poses, const float* d_pts, const uint8_t* d_cols,
                                const uint64_t* offs, int32_t freespace, int32_t slot) {
  return prepare_job(L, cfg, F, poses, d_pts, d_cols, offs, freespace, slot, nullptr);
}

int32_t cg_prepare_batch_staged(cg_layer* L, const cg_integrator_config* cfg, size_t F,
                                const float* poses, int32_t stage_slot, const uint64_t* offs,
                                int32_t freespace, int32_t slot) {
  StagedInputs in;
  const int32_t rc = staged_inputs("cg_prepare_batch_staged", L, cfg, poses, stage_slot, F, offs, &in);
  if (rc) return rc;
  return prepare_job(L, cfg, F, poses, in.pts, in.cols, offs, freespace, slot, in.ready);
}

int32_t cg_integrate_prepared(cg_layer* L, int32_t slot, cg_integrate_stats* stats) {
  if (!L || slot < 0 || slot > 1 || !L->ctx->prepared[slot].valid) {
    set_error("cg_integrate_prepared: nothing prepared in this slot");
    return CG_ERR_INVALID_ARG;
  }
  cg_context* ctx = L->ctx;
  cg_context::PreparedJob& pj = ctx->prepared[slot];
  pj.valid = false;
  // a front half queued for another voxel size is dropped unread
  const bool usable = pj.front_queued && pj.voxel_size == L->v.voxel_size;
  return integrate_job(L, &pj.cfg, pj.offs.size() - 1, pj.poses.data(), pj.d_points, pj.d_colors,
                       pj.offs.data(), pj.freespace, stats, usable ? &ctx->prep[slot] : nullptr,
                       ctx->prep_done[slot], pj.inputs_ready);
}

void cg_integrator_config_default(cg_integrator_config* c) {
  if (!c) return;
  c->default_truncation_distance = 0.1f;
  c->max_weight = 10000.0f;
  c->voxel_carving_enabled = 1;
  c->min_ray_length_m = 0.1f;
  c->max_ray_length_m = 5.0f;
  c->use_const_weight = 0;
  c->allow_clear = 1;
  c->use_weight_dropoff = 1;
  c->use_sparsity_compensation_factor = 0;
  c->sparsity_compensation_factor = 1.0f;
  c->enable_anti_grazing = 0;
  c->method = CG_METHOD_MERGED;
  c->integration_order_mode = CG_ORDER_MIXED;
  c->start_voxel_subsampling_factor = 2.0f;
  c->max_consecutive_ray_collisions = 2;
}

int32_t cg_integrate_batch_device(cg_layer* L, const cg_integrator_config* cfg, size_t F,
                                  const float* poses, const float* d_pts, const uint8_t* d_cols,
                                  const uint64_t* offs, int32_t freespace,
                                  cg_integrate_stats* stats) {
  return integrate_job(L, cfg, F, poses, d_pts, d_cols, offs, freespace, stats);
}

int32_t cg_integrate_batch(cg_layer* L, const cg_integrator_config* cfg, size_t F,
                           const float* poses, const float* pts, const uint8_t* cols,
                           const uint64_t* offs, int32_t freespace, cg_integrate_stats* stats) {
  if (!L || !cfg || !poses || !offs) {
    set_error("cg_integrate: null argument");
    return CG_ERR_INVALID_ARG;
  }
  const size_t first = offs[0], total = offs[F] - offs[0];
  if (total && (!pts || !cols)) {
    set_error("cg_integrate: null argument");
    return CG_ERR_INVALID_ARG;
  }
  std::vector<uint64_t> rel(F + 1);
  for (size_t f = 0; f <= F; ++f) rel[f] = offs[f] - first;
  cg_context* ctx = L->ctx;
  int32_t rc = stage_inputs(ctx, pts + 3 * first, cols + 4 * first, total);
  if (rc) return rc;
  return cg_integrate_batch_device(L, cfg, F, poses, ctx->points.as<float>(),
                                   ctx->colors.as<uint8_t>(), rel.data(), freespace, stats);
}

int32_t cg_stage_batch_async(cg_context* ctx, int32_t slot, const float* pts, const uint8_t* cols,
                             size_t n) {
  if (!ctx || slot < 0 || slot > 1 || (n && (!pts || !cols))) {
    set_error("cg_stage_batch_async: invalid argument");
    return CG_ERR_INVALID_ARG;
  }
  CG_CUDA(cudaSetDevice(ctx->device));
  if (!ctx->copy_stream)
    CG_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
  if (!ctx->stage_ready[slot])
    CG_CUDA(cudaEventCreateWithFlags(&ctx->stage_ready[slot], cudaEventDisableTiming));
  CG_CUDA(ctx->stage_pts[slot].reserve(n * 3 * sizeof(float)));
  CG_CUDA(ctx->stage_cols[slot].reserve(n * 4));
  if (n) {
    CG_CUDA(cudaMemcpyAsync(ctx->stage_pts[slot].p, pts, n * 3 * sizeof(float),
                            cudaMemcpyHostToDevice, ctx->copy_stream));
    CG_CUDA(cudaMemcpyAsync(ctx->stage_cols[slot].p, cols, n * 4, cudaMemcpyHostToDevice,
                            ctx->copy_stream));
  }
  CG_CUDA(cudaEventRecord(ctx->stage_ready[slot], ctx->copy_stream));
  ctx->stage_points[slot] = n;
  return CG_OK;
}

int32_t cg_integrate_batch_staged(cg_layer* L, const cg_integrator_config* cfg, size_t F,
                                  const float* poses, int32_t slot, const uint64_t* offs,
                                  int32_t freespace, cg_integrate_stats* stats) {
  StagedInputs in;
  const int32_t rc = staged_inputs("cg_integrate_batch_staged", L, cfg, poses, slot, F, offs, &in);
  if (rc) return rc;
  CG_CUDA(cudaStreamWaitEvent(L->ctx->stream, in.ready, 0));
  return cg_integrate_batch_device(L, cfg, F, poses, in.pts, in.cols, offs, freespace, stats);
}

int32_t cg_integrate_pointcloud_device(cg_layer* L, const cg_integrator_config* cfg,
                                       const float T[7], const float* d_pts, const uint8_t* d_cols,
                                       size_t n, int32_t freespace, cg_integrate_stats* stats) {
  const uint64_t offs[2] = {0, n};
  return cg_integrate_batch_device(L, cfg, 1, T, d_pts, d_cols, offs, freespace, stats);
}

int32_t cg_integrate_pointcloud(cg_layer* L, const cg_integrator_config* cfg, const float T[7],
                                const float* pts, const uint8_t* cols, size_t n, int32_t freespace,
                                cg_integrate_stats* stats) {
  const uint64_t offs[2] = {0, n};
  return cg_integrate_batch(L, cfg, 1, T, pts, cols, offs, freespace, stats);
}

}  // extern "C"
