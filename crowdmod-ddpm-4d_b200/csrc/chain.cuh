// The reverse chain x_T -> x_0 (models/diffusion/ddpm.py:206-282) shared by both backbones: the reverse-step update
// each backbone fuses into the last kernel of its denoiser evaluation, and the host driver that runs the T steps
// eagerly, as a captured step replayed T times, or as one whole-chain graph.
#pragma once
#include <functional>
#include <vector>

#include "../../include/crowdmod_b200.h"
#include "common.cuh"

namespace cm {

// ---- the reverse-step update (DDPM.step / DDIM, ddpm.py:25-38, :262-265; Sparsity guidance, guidance.py:4-8) ----
struct ReverseStep {
  float* x;              // [B][C][H][W][F] in/out; nullptr -> eps only, no update
  const float* coef;     // [nsteps][8] per-step coefficients (cm_chain_args)
  const int* step_dev;   // device step index
  int mode;              // 0 = DDPM, 1 = DDIM
  const float* noise;    // [nsteps][B*C*H*W*F] or nullptr -> Philox
  const unsigned long long* chain_dev;   // device {seed, sample_offset}: a new seed / shard offset needs no new graph
  float* history;        // optional [nsteps+1][B*C*H*W*F]; slot step+1 written
};

// One (sample b, site) of x and its C <= 4 channels, given the denoiser output eps[c]: element e0 + c * plane with
// e0 = b * C * plane + site, site = (row * W + col) * F + frame.  z is injected or one Philox4x32-10 draw (counter =
// global sample index * plane + site, step; key = seed: invariant to how the batch is sharded over GPUs).
__device__ __forceinline__ void reverse_step_update(const ReverseStep& r, const float* eps, int C, int B, int b,
                                                    size_t plane, size_t site) {
  const int step = *r.step_dev;
  const float* cf = r.coef + (size_t)step * 8;
  const size_t e0 = ((size_t)b * C) * plane + site;
  const size_t nelem = (size_t)B * C * plane;
  float z[4] = {0.f, 0.f, 0.f, 0.f};
  const float zc = (r.mode == 0) ? cf[2] : cf[4];
  if (zc != 0.f) {
    if (r.noise) {
#pragma unroll
      for (int c = 0; c < C; ++c) z[c] = r.noise[(size_t)step * nelem + e0 + c * plane];
    } else {
      const unsigned long long seed = r.chain_dev[0];
      const long long soff = static_cast<long long>(r.chain_dev[1]);
      const unsigned long long gp = ((unsigned long long)(soff + b)) * (unsigned long long)plane + site;
      const uint4 rnd = philox4x32_10(make_uint4((uint32_t)gp, (uint32_t)(gp >> 32), (uint32_t)step, 0u),
                                      make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
      const float2 n0 = box_muller(rnd.x, rnd.y), n1 = box_muller(rnd.z, rnd.w);
      z[0] = n0.x; z[1] = n0.y; z[2] = n1.x; z[3] = n1.y;
    }
  }
#pragma unroll
  for (int c = 0; c < C; ++c) {
    const size_t e = e0 + c * plane;
    const float xv = r.x[e];
    float xn;
    if (r.mode == 0) {
      // ddpm.py:33-37: one_by_sqrt_alpha * (x - (beta/sqrt(1-abar)) * eps) + sqrt(beta) * z
      xn = cf[0] * (xv - cf[1] * eps[c]) + cf[2] * z[c];
    } else {
      // ddpm.py:262-265 (DDIM eq. 12)
      const float x0 = (xv - cf[0] * eps[c]) / cf[1];
      xn = cf[2] * x0 + cf[3] * eps[c] + cf[4] * z[c];
    }
    if (c == 0 && cf[5] != 0.f) {
      // guidance.py:4-8 + ddpm.py:223-226: x[:,0] -= lambda*sigma*sign(x[:,0])
      const float sg = (xn > 0.f) ? 1.f : ((xn < 0.f) ? -1.f : 0.f);
      xn -= cf[5] * sg;
    }
    r.x[e] = xn;
    if (r.history) r.history[(size_t)(step + 1) * nelem + e] = xn;
  }
}

// Op-level entry points (one kernel, one step): {seed, sample_offset, step} in a fresh device allocation *dev that
// rs.chain_dev / rs.step_dev point into, read from device memory as in a chain step.  The caller frees *dev.
int stage_step_state(ReverseStep& rs, unsigned long long** dev, unsigned long long seed, long long sample_offset,
                     int step, cudaStream_t st);

// ---- the chain driver ----
// Everything a chain reads at run time lives in buffers the driver owns (step index, timestep, schedule tables,
// Philox seed / shard offset) and the caller's staging copies of x / past, so one executable graph serves every
// chain of the same (n, nsteps, mode, noise, history, use_graph).
struct ChainDriver {
  int* d_step = nullptr;                     // [0] step index, [1] current timestep
  unsigned long long* d_chain = nullptr;     // [0] Philox seed, [1] sample offset
  int* d_tsteps = nullptr;
  float* d_coef = nullptr;
  int cap = 0;                               // steps d_tsteps / d_coef hold room for
  std::vector<int> tsteps_host;              // what d_tsteps / d_coef currently hold (re-uploaded only on change)
  std::vector<float> coef_host;
  cudaGraphExec_t graph_exec = nullptr;
  cm_chain_args graph_key{};
  int64_t graph_launches_per_step = 0;
  // the last chain
  int64_t launches = 0;                      // kernels enqueued
  int64_t graph_launches = 0;                // cudaGraphLaunch calls (1 whole-chain graph, nsteps per-step graph, 0 eager)
  int graph_rebuilt = 0;                     // whether the graph had to be (re)captured
};

// the cached graph bakes the caller's launches: drop it whenever they change (batch, buffers, parameter pointers)
void chain_drop_graph(ChainDriver& d);
void chain_free(ChainDriver& d);

// Enqueues one denoiser evaluation on `st` with the update `rs` fused into its last kernel, the timestep read from
// device memory at t_dev, and adds the kernels it enqueued to *launches.  Runs on the host only (eagerly or under
// stream capture).
using ChainStep = std::function<int(const ReverseStep& rs, const int* t_dev, cudaStream_t st, int64_t* launches)>;

// cm_chain_args semantics (include/crowdmod_b200.h): checks the arguments (tsteps inside [0, table_steps)), copies
// x / past into the staging buffers the step reads, runs the nsteps steps (each followed by the step advance) and
// copies x_0 back to a->x.  Nothing synchronises except an upload of changed schedule tables.
int chain_run(ChainDriver& d, const cm_chain_args& a, int table_steps, float* x_stage, size_t x_bytes,
              float* past_stage, size_t past_bytes, const ChainStep& step, cudaStream_t st);

}  // namespace cm
