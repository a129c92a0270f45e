// Weight / bias gradients of the field: dW_l = dY_l^T X_l and db_l = sum_points dY_l, accumulated over every
// 128-point tile of a pass.  SURVEY.md §2.4 K5 (bwd, wgrad), §8 rows a8, a9, a12.
//
// Replaces the autograd wgrad of every nn.Linear the reference evaluates per sample:
//   mlp_base.layers.0-7, field_output_{density,normals,roughness,diff,tint,bottleneck}, mlp_mid.layers.0,
//   field_output_mid            reflect_sampling_nerf_field.py:54-86 (forward at field.py:132-186)
//
// Operands are the block images the forward (X, csrc/field_fwd.cu stash) and the dgrad chain (dY,
// csrc/field_bwd.cu) left in HBM: [128 points][64 features] bf16 -- chunk-major images for everything the epilogues
// wrote (hidden activations, every dY block), 128-byte swizzled shared-memory images for the IPE / IDE encodings
// (csrc/field_layout.cuh).  Read "transposed" (MN-major UMMA descriptors, features contiguous: no-swizzle descriptors
// for the chunk-major blocks, SWIZZLE_128B ones for the encodings) they are directly the A = dY^T and B = X operands of
//   D[out, in] (+)= sum over 16 points  dY[pt, out] * X[pt, in]            (tcgen05.mma, fp32 in TMEM)
// One CTA owns one job = (layer, all <=256 output features, <=256 input features) and a contiguous range of
// tiles (split-K over points); its accumulators stay in TMEM for the whole range and are stored once into the CTA's
// slot of the caller's workspace; wgrad_reduce_kernel then adds the slots of every job into the blob in split order, so
// the gradient is the same from run to run.  db comes from the same shared-memory dY slabs, summed by the otherwise idle
// epilogue warps.
//
// HBM-bound: algorithmic bytes = (loaded dY blocks + n_blocks) * 16 KB per tile and job; 82 block reads = 1.31 MB per tile
// over the 12 active jobs (10.25 KB per point) against 2 * 618k * 128 = 158 MFLOP per tile.
//
// The bottleneck layer is linear in h7 (bott = h7 Wb^T + bb, no activation) and feeds only the mid layer, so neither the
// bottleneck activations nor their gradients are stashed: with G = dY_mid^T h7 (rows 64-191 of job 10, which multiplies
// [seed | dY_mid] with h7 in one pass) and db_mid,
//   dW_mid[:, bott part] = dY_mid^T bott     = G Wb^T + db_mid bb^T
//   dW_bott              = (dY_mid Wmb)^T h7 = Wmb^T G            db_bott = Wmb^T db_mid
// (rsn_field_wgrad_finish, once per step on the accumulated -- and all-reduced -- blob): 8 of the 95 block reads and 8 of the 80
// stash blocks per tile disappear from the wgrad, the training forward and the backward chain.
#include "field_wgrad_body.cuh"
#include <stdio.h>


extern "C" int64_t rsn_field_dy_stash_bytes(int64_t n_points) {
  return ((n_points + TILE - 1) / TILE) * (int64_t)DY_BLOCKS * BLOCK_BYTES;
}

// Float offsets of every job's dW / db region inside the gradient blob: out[2*j] = dW offset, out[2*j+1] = db
// offset or -1.  Returns the number of jobs; *total_floats = blob size.  HOST pointers.
extern "C" int rsn_field_wgrad_layout(int64_t* host_offsets, int64_t* host_shapes, int64_t* total_floats) {
  int64_t off = 0;
  for (int j = 0; j < kNumJobs; ++j) {
    const int m = kJobs[j].m_blocks * 64, n = kJobs[j].n_blocks * 64;
    if (host_offsets) host_offsets[2 * j] = off;
    if (host_shapes) host_shapes[2 * j] = m, host_shapes[2 * j + 1] = n;
    off += (int64_t)m * n;
    if (host_offsets) host_offsets[2 * j + 1] = kJobs[j].has_db ? off : -1;
    if (kJobs[j].has_db) off += m;
  }
  if (total_floats) *total_floats = off;
  return kNumJobs;
}

namespace {
constexpr int MID_IN = 290, MID_IDE = 34;   // mlp_mid.layers.0.weight is [128][34 IDE + 256 bottleneck]
// region 9 (dW_bott [256][256], db_bott [256]) from G (region 12 dW [128][256]) and db_mid: block j, thread k
__global__ void __launch_bounds__(256) wgrad_finish_bott_kernel(const float* __restrict__ G, const float* __restrict__ db_mid,
                                                                const float* __restrict__ w_mid, float* __restrict__ dw_bott,
                                                                float* __restrict__ db_bott) {
  __shared__ float wcol[128];   // Wmb[:, j]
  const int j = blockIdx.x, k = threadIdx.x;
  if (k < 128) wcol[k] = w_mid[k * MID_IN + MID_IDE + j];
  __syncthreads();
  float acc = 0.f;
#pragma unroll 8
  for (int m = 0; m < 128; ++m) acc = fmaf(wcol[m], G[m * 256 + k], acc);
  dw_bott[j * 256 + k] = acc;
  if (k == 0) {
    float b = 0.f;
    for (int m = 0; m < 128; ++m) b = fmaf(wcol[m], db_mid[m], b);
    db_bott[j] = b;
  }
}
// region 12: row m of dW_mid[:, bott part] = G[m, :] Wb^T + db_mid[m] bb, and db_mid itself: block m, thread j
__global__ void __launch_bounds__(256) wgrad_finish_mid_kernel(const float* __restrict__ G, const float* __restrict__ db_mid,
                                                               const float* __restrict__ w_bott, const float* __restrict__ b_bott,
                                                               float* __restrict__ dw_mid_bott, float* __restrict__ db_mid_out) {
  __shared__ float4 grow[64];
  const int m = blockIdx.x, j = threadIdx.x;
  if (j < 64) grow[j] = reinterpret_cast<const float4*>(G + m * 256)[j];
  __syncthreads();
  const float4* w = reinterpret_cast<const float4*>(w_bott + j * 256);
  float acc = db_mid[m] * b_bott[j];
#pragma unroll 8
  for (int k = 0; k < 64; ++k) {
    const float4 a = grow[k], b = __ldg(w + k);
    acc = fmaf(a.x, b.x, fmaf(a.y, b.y, fmaf(a.z, b.z, fmaf(a.w, b.w, acc))));
  }
  dw_mid_bott[m * 256 + j] = acc;
  if (j == 0) db_mid_out[m] = db_mid[m];
}
}  // namespace

// Completes the gradient blob after the last rsn_field_wgrad of a step (and after the all-reduce): fills the bottleneck
// layer's region and turns G into the bottleneck columns of the mid layer's weight gradient (see the header comment).
// w_bott [256][256], b_bott [256], w_mid [128][290]: the fp32 parameters (device).
extern "C" int rsn_field_wgrad_finish(float* grad_blob, const float* w_bott, const float* b_bott, const float* w_mid,
                                      cudaStream_t stream) {
  RSN_ARG(grad_blob && w_bott && b_bott && w_mid, "rsn_field_wgrad_finish: null pointer");
  RSN_ARG(((uintptr_t)grad_blob & 15) == 0 && ((uintptr_t)w_bott & 15) == 0, "rsn_field_wgrad_finish: 16-byte alignment");
  int64_t offs[2 * MAX_JOBS], total = 0;
  rsn_field_wgrad_layout(offs, nullptr, &total);
  const float* G = grad_blob + offs[2 * 10] + 64 * 256;          // rows 64-191 of job 10's [256][256] region
  const float* db_mid = grad_blob + offs[2 * 10 + 1] + 64;
  RSN_ARG((offs[2 * 10] & 3) == 0, "rsn_field_wgrad_finish: region 10 is not 16-byte aligned");
  wgrad_finish_bott_kernel<<<256, 256, 0, stream>>>(G, db_mid, w_mid, grad_blob + offs[2 * 9], grad_blob + offs[2 * 9 + 1]);
  RSN_LAUNCH_CHECK("wgrad_finish_bott_kernel");
  wgrad_finish_mid_kernel<<<128, 256, 0, stream>>>(G, db_mid, w_bott, b_bott, grad_blob + offs[2 * 12],
                                                   grad_blob + offs[2 * 12 + 1]);
  RSN_LAUNCH_CHECK("wgrad_finish_mid_kernel");
  return 0;
}

namespace {
constexpr int MAX_WGRAD_CTAS = 160;   // one wave on a B200 (148 SMs); bounds the workspace
}

extern "C" int64_t rsn_field_wgrad_workspace_bytes(void) {
  int64_t part_len = 0;
  for (int j = 0; j < kNumJobs; ++j) {
    const int64_t m = kJobs[j].m_blocks * 64;
    part_len = std::max(part_len, m * kJobs[j].n_blocks * 64 + (kJobs[j].has_db ? m : 0));
  }
  return (int64_t)MAX_WGRAD_CTAS * part_len * (int64_t)sizeof(float);
}

extern "C" int rsn_field_wgrad(const void* x_stash, const void* dy_stash, int64_t n_points, float* grad_blob,
                               void* workspace, const int* n_rays_dev, int64_t points_per_ray, cudaStream_t stream) {
  RSN_ARG(n_points >= 0, "rsn_field_wgrad: bad shape");
  RSN_ARG(!n_rays_dev || (points_per_ray >= 1 && points_per_ray < (1 << 20)), "rsn_field_wgrad: bad points_per_ray");
  if (n_points == 0) return 0;
  RSN_ARG(x_stash && dy_stash && grad_blob && workspace, "rsn_field_wgrad: null pointer");
  RSN_ARG(((uintptr_t)grad_blob & 15) == 0 && ((uintptr_t)workspace & 15) == 0,
          "rsn_field_wgrad: grad_blob and workspace must be 16-byte aligned");
  RSN_ARG(((uintptr_t)x_stash & 15) == 0 && ((uintptr_t)dy_stash & 15) == 0, "rsn_field_wgrad: stashes must be 16-byte aligned");
  WParams p;
  const int cta = fill_wgrad_params(p, x_stash, dy_stash, n_points, grad_blob, std::min(rsn_num_sms(), MAX_WGRAD_CTAS));
  p.part = (float*)workspace;
  p.n_rays_dev = n_rays_dev;
  p.pts_per_ray = n_rays_dev ? (int)points_per_ray : 1;
  const size_t smem = (size_t)RING_BYTES + 1024;
  static std::atomic<unsigned long long> done;
  RSN_CUDA(rsn_ensure_smem(field_wgrad_kernel, (int)smem, done));
  field_wgrad_kernel<<<cta, W_THREADS, smem, stream>>>(p);
  RSN_LAUNCH_CHECK("field_wgrad_kernel");
  wgrad_reduce_kernel<<<dim3(32, kNumJobs), 256, 0, stream>>>(p);
  RSN_LAUNCH_CHECK("wgrad_reduce_kernel");
  if (p.debug & 16) {
    static unsigned long long t[2][160];
    RSN_CUDA(cudaStreamSynchronize(stream));
    RSN_CUDA(cudaMemcpyFromSymbol(t, g_wgrad_times, sizeof(t)));
    unsigned long long t0 = ~0ull;
    for (int i = 0; i < cta; ++i) t0 = t[0][i] < t0 ? t[0][i] : t0;
    for (int j = 0; j < p.n_jobs; ++j) {
      if (!p.jobs[j].n_ctas) continue;
      unsigned long long lo = ~0ull, hi = 0;
      for (int i = p.jobs[j].cta_begin; i < p.jobs[j].cta_begin + p.jobs[j].n_ctas; ++i) {
        lo = t[1][i] < lo ? t[1][i] : lo;
        hi = t[1][i] > hi ? t[1][i] : hi;
      }
      fprintf(stderr, "wgrad job %2d: %2d CTAs, %d+%d blocks, CTAs end at %.1f .. %.1f us\n", j, p.jobs[j].n_ctas,
              p.jobs[j].a_load, p.jobs[j].n_blocks, (lo - t0) * 1e-3, (hi - t0) * 1e-3);
    }
  }
  return 0;
}
