// Body of the wgrad kernel (see field_wgrad.cu for the description).
#pragma once
#include "rsn_common.cuh"
#include "umma.cuh"
#include "field_layout.cuh"
#include <algorithm>
#include <stdlib.h>

namespace {

using namespace umma;
using namespace rsnf;

constexpr int W_THREADS = 192;      // warp 0 producer, warp 1 MMA issuer, warps 2-5 db + epilogue
#ifndef RSN_WGRAD_SLAB_ROWS
#define RSN_WGRAD_SLAB_ROWS 64
#endif
constexpr int SLAB_ROWS = RSN_WGRAD_SLAB_ROWS;   // points per pipeline slab (SLAB_ROWS / 16 K-steps)
constexpr int SLAB_BLOCK_BYTES = SLAB_ROWS * 128;
constexpr int RING_BYTES = 196608;                 // 192 KB ring of (m_blocks + n_blocks) * SLAB_BLOCK_BYTES stages:
constexpr int MAX_W_STAGES = 8;                    // 3 stages for the 4 + 4 block jobs, up to 8 for the small ones
constexpr int MAX_JOBS = 16;

struct WJob {
  int a_blk, m_blocks;   // first dY block of the job inside a dY tile; 2 (M=128) or 4 (M=256)
  int a_load;            // dY blocks actually loaded (m_blocks, or 3: the MMA's fourth A block is then the first X block)
  int b_blk, n_blocks;   // first X block inside a stash tile; 1, 2 or 4 (N = 64, 128, 256)
  int a_cm, b_cm;        // 1: the dY / X blocks are chunk-major images (field_layout.cuh), 0: swizzled images
  int out_off, db_off;   // float offsets into the gradient blob: dW [64 m_blocks][64 n_blocks], db or -1
  int cta_begin, n_ctas;
  int part_off, part_len;  // this job's partial sums in the workspace: split k at part_off + k * part_len floats (dW, then db)
};
struct WParams {
  const uint8_t* x;      // forward stash  [n_tiles][STASH_BLOCKS][16 KB]
  const uint8_t* dy;     // dgrad stash    [n_tiles][DY_BLOCKS][16 KB]
  int n_tiles;           // capacity when n_rays_dev is set
  const int* n_rays_dev; // optional device-side ray count (bounce passes): tiles = ceil(min(*n_rays_dev, rays) * pts_per_ray / 128)
  int pts_per_ray;
  float* grad;
  float* part;           // workspace: every CTA's partial dW / db, added into grad in split order by wgrad_reduce_kernel
  int n_jobs;
  int debug;   // RSN_WGRAD_DEBUG (test build only): 1 = MMA only (no loads, no db), 2 = loads only (no MMA)
  WJob jobs[MAX_JOBS];
};

// RSN_WGRAD_DEBUG & 16: start / end %globaltimer of every CTA (per-job balance diagnostics)
__device__ unsigned long long g_wgrad_times[2][160];

struct WBarriers {
  uint64_t full[MAX_W_STAGES], empty[MAX_W_STAGES];
  uint64_t acc_full;
  uint32_t tmem_slot;
};

__device__ __forceinline__ void wgrad_body(const WParams& p) {
  const int vbid = (int)blockIdx.x;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  __shared__ WBarriers bars;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if ((p.debug & 16) && threadIdx.x == 0 && vbid < 160) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    g_wgrad_times[0][vbid] = t;
  }

  int j = 0;
  for (int i = 0; i < p.n_jobs; ++i)
    if (vbid >= p.jobs[i].cta_begin && vbid < p.jobs[i].cta_begin + p.jobs[i].n_ctas) j = i;
  const WJob job = p.jobs[j];
  const int split = vbid - job.cta_begin;
  int n_tiles = p.n_tiles;
  if (p.n_rays_dev) {
    const int64_t pts = (int64_t)max(__ldg(p.n_rays_dev), 0) * p.pts_per_ray;
    n_tiles = (int)min((int64_t)n_tiles, (pts + TILE - 1) / TILE);
  }
  // tiles split, split + n_ctas, ...: the CTAs of a job stream neighbouring tiles at the same time
  const bool interleave = !(p.debug & 8);
  const int t0 = interleave ? split : (int)(((int64_t)n_tiles * split) / job.n_ctas);
  const int t1 = interleave ? n_tiles : (int)(((int64_t)n_tiles * (split + 1)) / job.n_ctas);
  const int tstep = interleave ? job.n_ctas : 1;
  // mb = dY blocks loaded per slab; m_out = 64-row blocks of the accumulator (2 or 4).  mb = 3, m_out = 4: the second M=128
  // MMA reads blocks 2 and "3" = the first X block, which sits right behind the dY blocks in the stage -- its 64 output rows
  // are a finite by-product nobody reads, and no fourth dY block has to be fetched
  const int mb = job.a_load, m_out = job.m_blocks, nb = job.n_blocks;
  // a job with fewer blocks per slab gets more stages: the same bytes in flight for every CTA
  const int SLAB_BYTES = (mb + nb) * SLAB_BLOCK_BYTES;
  const int W_STAGES = min(MAX_W_STAGES, RING_BYTES / SLAB_BYTES);
  const int n_slabs = (t1 > t0 ? (t1 - t0 + tstep - 1) / tstep : 0) * (TILE / SLAB_ROWS);

  if (warp == 1) {
    if (lane == 0) {
      for (int i = 0; i < MAX_W_STAGES; ++i) {
        mbar_init(&bars.full[i], 1);
        mbar_init(&bars.empty[i], 1 + 4);   // tcgen05.commit + one arrival per db warp
      }
      mbar_init(&bars.acc_full, 1);
      fence_barrier_init();
    }
    __syncwarp();
    tmem_alloc(&bars.tmem_slot, 512);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = bars.tmem_slot;

  if (warp == 0) {
    if (lane == 0 && (p.debug & 3) != 1) {
      int stage = 0;
      uint32_t phase = 0;
      for (int t = t0; t < t1; t += tstep) {
        const uint8_t* dyt = p.dy + ((size_t)t * DY_BLOCKS + job.a_blk) * BLOCK_BYTES;
        const uint8_t* xt = p.x + (size_t)t * STASH_TILE_BYTES + (size_t)job.b_blk * BLOCK_BYTES;
        for (int s = 0; s < TILE / SLAB_ROWS; ++s) {
          mbar_wait(&bars.empty[stage], phase ^ 1);
          mbar_expect_tx(&bars.full[stage], (uint32_t)(mb + nb) * SLAB_BLOCK_BYTES);
          uint8_t* dst = smem + (size_t)stage * SLAB_BYTES;
          for (int i = 0; i < mb; ++i)
            bulk_g2s(dst + i * SLAB_BLOCK_BYTES, dyt + (size_t)i * BLOCK_BYTES + s * SLAB_BLOCK_BYTES,
                     SLAB_BLOCK_BYTES, &bars.full[stage]);
          for (int i = 0; i < nb; ++i)
            bulk_g2s(dst + (mb + i) * SLAB_BLOCK_BYTES, xt + (size_t)i * BLOCK_BYTES + s * SLAB_BLOCK_BYTES,
                     SLAB_BLOCK_BYTES, &bars.full[stage]);
          if (++stage == W_STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // (whole warp: control flow and barrier waits; tcgen05.mma / tcgen05.commit under elect_one_sync(), see umma.cuh)
    if (n_slabs > 0) {
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t idesc = instr_desc_bf16(128, nb * 64, 1, 1);
      for (int s = 0; s < n_slabs; ++s) {
        if ((p.debug & 3) != 1) mbar_wait(&bars.full[stage], phase);
        tc_fence_after();
        const uint32_t base = smem_u32(smem + (size_t)stage * SLAB_BYTES);
        // MN-major operands (the 64 features of a block are the contiguous dimension), two block images:
        //   swizzled    (128-byte swizzle): LBO = stride between the 64-feature blocks of the slab, SBO = 1024 (8 points);
        //               one K = 16 step (16 points) advances the start address by 2048 bytes
        //   chunk-major (no swizzle): core matrix = 8 points x 16 B = 128 contiguous bytes; LBO = 128 (next 8 points),
        //               SBO = 1024 (next 8 features -- across the slab's blocks too: 8 chunks x 1024 B = one block);
        //               one K = 16 step advances the start address by 256 bytes
        const uint32_t a_hi = job.a_cm ? desc_hi_noswz(STASH_CHUNK_STRIDE) : desc_hi_sw128(1024);
        const uint32_t b_hi = job.b_cm ? desc_hi_noswz(STASH_CHUNK_STRIDE) : desc_hi_sw128(1024);
        const uint32_t a_lo = desc_lo(base, job.a_cm ? 128 : SLAB_BLOCK_BYTES);
        const uint32_t b_lo = desc_lo(base + mb * SLAB_BLOCK_BYTES, job.b_cm ? 128 : SLAB_BLOCK_BYTES);
        const uint32_t a_ks = job.a_cm ? 16u : 128u, b_ks = job.b_cm ? 16u : 128u;   // K-step advance in 16-byte units
        if ((p.debug & 3) != 2 && elect_one_sync()) {
          // all K-steps of the slab into one accumulator, then the other: interleaving the two accumulators MMA by
          // MMA is measurably slower (2.6 vs 4.2 ms for the MMA stream alone at C2)
#pragma unroll
          for (int ks = 0; ks < SLAB_ROWS / 16; ++ks)
            mma_bf16_ss_lo2(tmem, a_lo + ks * a_ks, a_hi, b_lo + ks * b_ks, b_hi, idesc, (s | ks) != 0);
          if (m_out == 4) {
#pragma unroll
            for (int ks = 0; ks < SLAB_ROWS / 16; ++ks)
              mma_bf16_ss_lo2(tmem + 256, a_lo + (2 * SLAB_BLOCK_BYTES >> 4) + ks * a_ks, a_hi, b_lo + ks * b_ks, b_hi, idesc,
                              (s | ks) != 0);
          }
        }
        if (elect_one_sync()) mma_commit(&bars.empty[stage]);
        if (++stage == W_STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
      if (elect_one_sync()) mma_commit(&bars.acc_full);
    }
  } else {
    // ---- db: column sums of the dY slabs while they sit in shared memory; then the dW flush.
    // The dY blocks are chunk-major images: inside a slab block the 16-byte chunk c (8 features) of point r sits at
    // c * 1024 + r * 16.  Warp w sums block w; lane = point (r = lane, lane + 32), so every 128-bit shared load of a warp
    // reads 512 contiguous bytes (conflict-free); 8 chunks x 8 features = 64 partial sums per thread, reduced across the
    // lanes once at the end.
    static_assert(DY_CHUNK_MAJOR && SLAB_ROWS == 64, "db sums are written for chunk-major dY slabs of 64 points");
    const int blk = warp - 2;
    const bool db_active = blk < mb;
    float acc[8][8];
#pragma unroll
    for (int c = 0; c < 8; ++c)
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[c][i] = 0.f;
    int stage = 0;
    uint32_t phase = 0;
    for (int s = 0; s < ((p.debug & 3) == 1 ? 0 : n_slabs); ++s) {
      mbar_wait(&bars.full[stage], phase);
      if (db_active && (p.debug & 3) != 3) {
        const uint32_t src = smem_u32(smem + (size_t)stage * SLAB_BYTES) + blk * SLAB_BLOCK_BYTES + (uint32_t)lane * 16u;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          uint4 v[8];
#pragma unroll
          for (int c = 0; c < 8; ++c)
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                         : "=r"(v[c].x), "=r"(v[c].y), "=r"(v[c].z), "=r"(v[c].w)
                         : "r"(src + (uint32_t)c * STASH_CHUNK_STRIDE + (uint32_t)h * 512u));
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            acc[c][0] += __uint_as_float(v[c].x << 16), acc[c][1] += __uint_as_float(v[c].x & 0xffff0000u);
            acc[c][2] += __uint_as_float(v[c].y << 16), acc[c][3] += __uint_as_float(v[c].y & 0xffff0000u);
            acc[c][4] += __uint_as_float(v[c].z << 16), acc[c][5] += __uint_as_float(v[c].z & 0xffff0000u);
            acc[c][6] += __uint_as_float(v[c].w << 16), acc[c][7] += __uint_as_float(v[c].w & 0xffff0000u);
          }
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars.empty[stage]);
      if (++stage == W_STAGES) {
        stage = 0;
        phase ^= 1;
      }
    }
    if (n_slabs > 0) {
      if (db_active && job.db_off >= 0 && (p.debug & 3) != 1) {
        // feature c * 8 + i of the block: summed over the lanes, kept by lane (c * 8 + i) & 31 in mine[(c * 8 + i) >> 5]
        float mine[2] = {0.f, 0.f};
#pragma unroll
        for (int c = 0; c < 8; ++c)
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float t = warp_sum(acc[c][i]);
            if (lane == ((c * 8 + i) & 31)) mine[(c * 8 + i) >> 5] = t;
          }
        float* db = p.part + job.part_off + (size_t)split * job.part_len + m_out * 64 * nb * 64 + blk * 64;
        db[lane] = mine[0];
        db[32 + lane] = mine[1];
      }
      mbar_wait(&bars.acc_full, 0);
      tc_fence_after();
      const int q = warp & 3;
      const int row = q * 32 + lane;
      const int N = nb * 64;
      for (int h = 0; h < ((p.debug & 4) ? 0 : m_out / 2); ++h) {
        float* out = p.part + job.part_off + (size_t)split * job.part_len + (size_t)(h * 128 + row) * N;
        for (int c0 = 0; c0 < N; c0 += 32) {
          uint32_t v[32];
          tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + h * 256 + c0, v);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 32; i += 4)
            *reinterpret_cast<float4*>(out + c0 + i) = make_float4(__uint_as_float(v[i]), __uint_as_float(v[i + 1]),
                                                                   __uint_as_float(v[i + 2]), __uint_as_float(v[i + 3]));
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 512);
  if ((p.debug & 16) && threadIdx.x == 0 && vbid < 160) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    g_wgrad_times[1][vbid] = t;
  }
}

__global__ void __launch_bounds__(W_THREADS, 1) field_wgrad_kernel(const __grid_constant__ WParams p) {
  wgrad_body(p);
}

// Adds the partial sums of every job's CTAs into the gradient blob, in split order: the same fp32 sums every run.
// grid (blocks, jobs); a CTA that had no tile wrote nothing and is skipped; db rows past the loaded dY blocks are not
// written by the wgrad (the blob keeps its value there, as it did with atomics).
__global__ void __launch_bounds__(256) wgrad_reduce_kernel(const __grid_constant__ WParams p) {
  const WJob job = p.jobs[blockIdx.y];
  if (job.n_ctas == 0 || (p.debug & 4)) return;
  int n_tiles = p.n_tiles;
  if (p.n_rays_dev) {
    const int64_t pts = (int64_t)max(__ldg(p.n_rays_dev), 0) * p.pts_per_ray;
    n_tiles = (int)min((int64_t)n_tiles, (pts + TILE - 1) / TILE);
  }
  const bool interleave = !(p.debug & 8);
  const int dw = job.m_blocks * 64 * job.n_blocks * 64;
  const int db_rows = (job.db_off >= 0 && (p.debug & 3) != 1) ? job.a_load * 64 : 0;
  for (int e = (blockIdx.x * blockDim.x + threadIdx.x) * 4; e < dw + db_rows; e += gridDim.x * blockDim.x * 4) {
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int k = 0; k < job.n_ctas; ++k) {
      const int t0 = interleave ? k : (int)(((int64_t)n_tiles * k) / job.n_ctas);
      const int t1 = interleave ? n_tiles : (int)(((int64_t)n_tiles * (k + 1)) / job.n_ctas);
      if (t1 <= t0) continue;
      const float4 v = *reinterpret_cast<const float4*>(p.part + job.part_off + (size_t)k * job.part_len + e);
      s.x += v.x, s.y += v.y, s.z += v.z, s.w += v.w;
    }
    float4* g = reinterpret_cast<float4*>(p.grad + job.out_off + e);     // db follows dW in the blob, as in the workspace
    float4 o = *g;
    o.x += s.x, o.y += s.y, o.z += s.z, o.w += s.w;
    *g = o;
  }
}

// The 12 jobs of one pass.  Gradient blob regions (fp32): dW [64 m_blocks][64 n_blocks] row-major, then db.
struct JobSpec {
  int a_blk, m_blocks, b_blk, n_blocks, has_db;
  int active = 1;   // 0: the region is part of the blob but filled by rsn_field_wgrad_finish, not by the kernel
  int a_load = 0;   // dY blocks to load if fewer than m_blocks (see wgrad_body); 0 = m_blocks
  int cost = 1000;  // measured time per loaded block of one CTA, relative to the 4 + 4 block jobs (x 1000): the small-slab jobs
                    // pay more per byte (RSN_WGRAD_DEBUG=16 prints when each job's CTAs finish)
};
const JobSpec kJobs[] = {
    {DY_H + 0, 4, STASH_ENC, 2, 1, 1, 0, 910},  //  0  layer 0            x enc
    {DY_H + 4, 4, STASH_H + 0, 4, 1},           //  1  layer 1            x h0
    {DY_H + 8, 4, STASH_H + 4, 4, 1},           //  2  layer 2            x h1
    {DY_H + 12, 4, STASH_H + 8, 4, 1},          //  3  layer 3            x h2
    {DY_H + 16, 4, STASH_ENC, 2, 0, 1, 0, 910}, //  4  layer 4 (enc part) x enc
    {DY_H + 16, 4, STASH_H + 12, 4, 1},         //  5  layer 4 (hidden)   x h3
    {DY_H + 20, 4, STASH_H + 16, 4, 1},         //  6  layer 5            x h4
    {DY_H + 24, 4, STASH_H + 20, 4, 1},         //  7  layer 6            x h5
    {DY_H + 28, 4, STASH_H + 24, 4, 1},         //  8  layer 7            x h6
    {DY_BOTT, 4, STASH_H + 28, 4, 1, 0},        //  9  bottleneck         x h7: derived from job 12 (rsn_field_wgrad_finish)
    {DY_SEED, 4, STASH_H + 28, 4, 1, 1, 3, 1100},  // 10  [seed | dY_mid] x h7: rows 16-31 heads, rows 64-191 G = dY_mid^T h7
    {DY_SEED, 2, STASH_MIDH, 2, 0, 1, 0, 990},  // 11  rgb (rows 0-15)    x mid hidden (db from job 10's sums)
    {DY_MID, 2, STASH_BOTT, 4, 1, 0},           // 12  mid x bottleneck: derived from job 10's G (rsn_field_wgrad_finish)
    {DY_MID, 2, STASH_IDE, 1, 0, 1, 0, 1160},   // 13  mid (IDE part)     x IDE
};
constexpr int kNumJobs = sizeof(kJobs) / sizeof(kJobs[0]);
static_assert(kNumJobs <= MAX_JOBS, "job table too small");
static_assert(SLAB_ROWS == STASH_SLAB_ROWS, "the chunk-major image is laid out in the wgrad's slabs");

// Job table of one pass for `cta_budget` wgrad CTAs: CTAs per job proportional to the job's bytes per tile (the kernel
// is HBM-bound).  Returns the number of CTAs used (<= cta_budget, one wave).
inline int fill_wgrad_params(WParams& p, const void* x_stash, const void* dy_stash, int64_t n_points, float* grad_blob,
                             int cta_budget) {
  p.x = (const uint8_t*)x_stash;
  p.dy = (const uint8_t*)dy_stash;
  p.n_tiles = (int)((n_points + TILE - 1) / TILE);
  p.grad = grad_blob;
  p.n_jobs = kNumJobs;
  p.debug = rsn_env_int("RSN_WGRAD_DEBUG", 0);
  p.n_rays_dev = nullptr;
  p.pts_per_ray = 1;
  int n_of[kNumJobs], used = 0;
  // CTAs per job proportional to the job's cost per tile = loaded blocks x measured relative time per block; the kernel
  // ends with the job whose CTAs carry the most, so the CTAs left over by the rounding go, one at a time, to the job with
  // the largest cost per CTA
  auto cost_of = [](int j) -> double {
    const JobSpec& k = kJobs[j];
    return k.active ? ((k.a_load ? k.a_load : k.m_blocks) + k.n_blocks) * (k.cost * 1e-3) : 0.0;
  };
  double total_cost = 0.0;
  for (int j = 0; j < kNumJobs; ++j) total_cost += cost_of(j);
  for (int j = 0; j < kNumJobs; ++j) {
    n_of[j] = kJobs[j].active ? std::min(std::max(1, (int)(cost_of(j) * cta_budget / total_cost)), p.n_tiles) : 0;
    used += n_of[j];
  }
  while (used < cta_budget) {
    int best = -1;
    double worst = 0.0;
    for (int j = 0; j < kNumJobs; ++j) {
      if (!kJobs[j].active) continue;
      const double load = cost_of(j) / n_of[j];
      if (n_of[j] < p.n_tiles && load > worst) worst = load, best = j;
    }
    if (best < 0) break;
    ++n_of[best];
    ++used;
  }
  int64_t off = 0, part = 0;
  int cta = 0;
  for (int j = 0; j < kNumJobs; ++j) {
    WJob& w = p.jobs[j];
    w.a_blk = kJobs[j].a_blk, w.m_blocks = kJobs[j].m_blocks, w.b_blk = kJobs[j].b_blk, w.n_blocks = kJobs[j].n_blocks;
    w.a_load = kJobs[j].a_load ? kJobs[j].a_load : kJobs[j].m_blocks;
    // block images (field_layout.cuh): the encodings are stashed as they sit in shared memory (swizzled), everything the
    // epilogues produce is chunk-major
    w.a_cm = DY_CHUNK_MAJOR ? 1 : 0;
    w.b_cm = (kJobs[j].b_blk == STASH_ENC || kJobs[j].b_blk == STASH_IDE) ? 0 : 1;
    w.out_off = (int)off;
    off += (int64_t)w.m_blocks * 64 * w.n_blocks * 64;
    w.db_off = kJobs[j].has_db ? (int)off : -1;
    if (kJobs[j].has_db) off += w.m_blocks * 64;
    w.cta_begin = cta, w.n_ctas = n_of[j];
    w.part_len = w.m_blocks * 64 * w.n_blocks * 64 + (kJobs[j].has_db ? w.m_blocks * 64 : 0);
    w.part_off = (int)part;
    part += (int64_t)n_of[j] * w.part_len;
    cta += n_of[j];
  }
  return cta;
}

}  // namespace
