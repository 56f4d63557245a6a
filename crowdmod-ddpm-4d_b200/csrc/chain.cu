// Reverse-chain driver shared by the UNet (cm_ddpm_sample) and DiT (cm_dit_sample) plans: chain.cuh.
#include <string.h>

#include "chain.cuh"

namespace cm {
namespace {

// ---- chain bookkeeping kernels ----
// step += 1; t_dev = tsteps[step]
__global__ void advance_step_kernel(int* step_dev, int* t_dev, const int* tsteps, int nsteps) {
  const int s = *step_dev + 1;
  *step_dev = s;
  *t_dev = tsteps[s < nsteps ? s : nsteps - 1];
}
int advance_step_enqueue(int* step_dev, int* t_dev, const int* tsteps, int nsteps, cudaStream_t st) {
  advance_step_kernel<<<1, 1, 0, st>>>(step_dev, t_dev, tsteps, nsteps);
  CM_CUDA(cudaGetLastError());
  return 0;
}
// same, as the last node of a conditional WHILE body: also sets the loop condition (step < nsteps)
__global__ void advance_step_cond_kernel(int* step_dev, int* t_dev, const int* tsteps, int nsteps,
                                         cudaGraphConditionalHandle h) {
  const int s = *step_dev + 1;
  *step_dev = s;
  *t_dev = tsteps[s < nsteps ? s : nsteps - 1];
  cudaGraphSetConditional(h, s < nsteps ? 1u : 0u);
}
int advance_step_cond_enqueue(int* step_dev, int* t_dev, const int* tsteps, int nsteps, cudaGraphConditionalHandle h,
                              cudaStream_t st) {
  advance_step_cond_kernel<<<1, 1, 0, st>>>(step_dev, t_dev, tsteps, nsteps, h);
  CM_CUDA(cudaGetLastError());
  return 0;
}
// start of a chain: step = 0, t_dev = tsteps[0], chain_dev = {seed, sample_offset} (arguments travel as
// kernel parameters: no host staging buffer, no synchronisation)
__global__ void chain_begin_kernel(int* step_dev, int* t_dev, const int* tsteps, unsigned long long* chain_dev,
                                   unsigned long long seed, long long sample_offset) {
  *step_dev = 0;
  *t_dev = tsteps[0];
  chain_dev[0] = seed;
  chain_dev[1] = static_cast<unsigned long long>(sample_offset);
}
int chain_begin_enqueue(int* step_dev, int* t_dev, const int* tsteps, unsigned long long* chain_dev,
                        unsigned long long seed, long long sample_offset, cudaStream_t st) {
  chain_begin_kernel<<<1, 1, 0, st>>>(step_dev, t_dev, tsteps, chain_dev, seed, sample_offset);
  CM_CUDA(cudaGetLastError());
  return 0;
}

// Captures one step + advance (use_graph 1: replayed nsteps times) or the same as the body of a conditional WHILE
// node whose condition the advance kernel sets from the device step counter (use_graph 2: the whole T-step loop is
// ONE graph launch, ddpm.py:214-231).
int capture(ChainDriver& d, const cm_chain_args& a, const ReverseStep& rs, const ChainStep& step) {
  int* t_dev = d.d_step + 1;
  int64_t per_step = 0;
  cudaStream_t cs;
  CM_CUDA(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
  cudaGraph_t g = nullptr;
  int e = 0;
  cudaError_t ce = cudaSuccess;
  if (a.use_graph == 1) {
    ce = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
    if (ce == cudaSuccess) {
      e = step(rs, t_dev, cs, &per_step);
      if (!e) e = advance_step_enqueue(d.d_step, t_dev, d.d_tsteps, a.nsteps, cs);
      ++per_step;
      ce = cudaStreamEndCapture(cs, &g);
    }
  } else {
    cudaGraphConditionalHandle h;
    cudaGraph_t body = nullptr;
    ce = cudaGraphCreate(&g, 0);
    if (ce == cudaSuccess) ce = cudaGraphConditionalHandleCreate(&h, g, 1, cudaGraphCondAssignDefault);
    if (ce == cudaSuccess) {
      cudaGraphNodeParams np{};
      np.type = cudaGraphNodeTypeConditional;
      np.conditional.handle = h;
      np.conditional.type = cudaGraphCondTypeWhile;
      np.conditional.size = 1;
      cudaGraphNode_t node;
      ce = cudaGraphAddNode(&node, g, nullptr, 0, &np);
      if (ce == cudaSuccess) body = np.conditional.phGraph_out[0];
    }
    if (ce == cudaSuccess)
      ce = cudaStreamBeginCaptureToGraph(cs, body, nullptr, nullptr, 0, cudaStreamCaptureModeThreadLocal);
    if (ce == cudaSuccess) {
      e = step(rs, t_dev, cs, &per_step);
      if (!e) e = advance_step_cond_enqueue(d.d_step, t_dev, d.d_tsteps, a.nsteps, h, cs);
      ++per_step;
      cudaGraph_t done = nullptr;
      ce = cudaStreamEndCapture(cs, &done);
    }
  }
  cudaStreamDestroy(cs);
  if (e || ce != cudaSuccess) {
    if (g) cudaGraphDestroy(g);
    if (e) return e;
    CM_CUDA(ce);
  }
  CM_CUDA(cudaGraphInstantiate(&d.graph_exec, g, 0));
  cudaGraphDestroy(g);
  d.graph_key = a;
  d.graph_launches_per_step = per_step;
  d.graph_rebuilt = 1;
  return 0;
}

}  // namespace

int stage_step_state(ReverseStep& rs, unsigned long long** dev, unsigned long long seed, long long sample_offset,
                     int step, cudaStream_t st) {
  CM_CUDA(cudaMalloc(dev, 3 * sizeof(unsigned long long)));
  const unsigned long long h[3] = {seed, static_cast<unsigned long long>(sample_offset), static_cast<unsigned long long>(step)};
  rs.chain_dev = *dev;
  rs.step_dev = reinterpret_cast<const int*>(*dev + 2);   // low word of a little-endian 64-bit slot
  CM_CUDA(cudaMemcpyAsync(*dev, h, sizeof(h), cudaMemcpyHostToDevice, st));
  return 0;
}

void chain_drop_graph(ChainDriver& d) {
  if (d.graph_exec) {
    cudaGraphExecDestroy(d.graph_exec);
    d.graph_exec = nullptr;
  }
}

void chain_free(ChainDriver& d) {
  chain_drop_graph(d);
  cudaFree(d.d_step);
  cudaFree(d.d_chain);
  cudaFree(d.d_tsteps);
  cudaFree(d.d_coef);
  d = ChainDriver{};
}

int chain_run(ChainDriver& d, const cm_chain_args& a, int table_steps, float* x_stage, size_t x_bytes,
              float* past_stage, size_t past_bytes, const ChainStep& step, cudaStream_t st) {
  CM_CHECK(a.past && a.x && a.tsteps && a.coef, "null argument");
  CM_CHECK(a.nsteps >= 1 && a.n >= 1, "nsteps and n must be >= 1");
  CM_CHECK(a.mode == 0 || a.mode == 1, "mode must be 0 (DDPM) or 1 (DDIM)");
  CM_CHECK(a.use_graph >= 0 && a.use_graph <= 2, "use_graph must be 0 (eager), 1 (per-step graph) or 2 (whole-chain graph)");
  for (int i = 0; i < a.nsteps; ++i)
    CM_CHECK(a.tsteps[i] >= 0 && a.tsteps[i] < table_steps, "tsteps[%d]=%d out of range", i, a.tsteps[i]);
  if (!d.d_step) CM_CUDA(cudaMalloc(&d.d_step, 2 * sizeof(int)));
  if (!d.d_chain) CM_CUDA(cudaMalloc(&d.d_chain, 2 * sizeof(unsigned long long)));
  if (a.nsteps > d.cap) {
    cudaFree(d.d_tsteps);
    cudaFree(d.d_coef);
    CM_CUDA(cudaMalloc(&d.d_tsteps, a.nsteps * sizeof(int)));
    CM_CUDA(cudaMalloc(&d.d_coef, (size_t)a.nsteps * 8 * sizeof(float)));
    d.cap = a.nsteps;
    d.tsteps_host.clear();
    d.coef_host.clear();
    chain_drop_graph(d);
  }
  // schedule tables: uploaded only when they differ from what the device already holds (the host
  // vectors are the staging copies: the async copies read them, never the caller's arrays)
  {
    const bool same_t = (int)d.tsteps_host.size() == a.nsteps &&
                        memcmp(d.tsteps_host.data(), a.tsteps, a.nsteps * sizeof(int)) == 0;
    const bool same_c = (int)d.coef_host.size() == a.nsteps * 8 &&
                        memcmp(d.coef_host.data(), a.coef, (size_t)a.nsteps * 8 * sizeof(float)) == 0;
    if (!same_t || !same_c) {
      // the previous chain may still be reading the device tables; the copy is stream-ordered behind it.
      // The staging vectors are rewritten only here, after making sure the last upload has drained.
      CM_CUDA(cudaStreamSynchronize(st));
      d.tsteps_host.assign(a.tsteps, a.tsteps + a.nsteps);
      d.coef_host.assign(a.coef, a.coef + (size_t)a.nsteps * 8);
      CM_CUDA(cudaMemcpyAsync(d.d_tsteps, d.tsteps_host.data(), a.nsteps * sizeof(int), cudaMemcpyHostToDevice, st));
      CM_CUDA(cudaMemcpyAsync(d.d_coef, d.coef_host.data(), (size_t)a.nsteps * 8 * sizeof(float),
                              cudaMemcpyHostToDevice, st));
      CM_CUDA(cudaStreamSynchronize(st));
    }
  }
  CM_CUDA(cudaMemcpyAsync(x_stage, a.x, x_bytes, cudaMemcpyDeviceToDevice, st));
  if (past_bytes) CM_CUDA(cudaMemcpyAsync(past_stage, a.past, past_bytes, cudaMemcpyDeviceToDevice, st));
  int* t_dev = d.d_step + 1;
  if (int e = chain_begin_enqueue(d.d_step, t_dev, d.d_tsteps, d.d_chain, a.seed, a.sample_offset, st)) return e;

  const ReverseStep rs{x_stage, d.d_coef, d.d_step, a.mode, a.noise, d.d_chain, a.history};

  d.launches = 0;
  d.graph_launches = 0;
  d.graph_rebuilt = 0;
  if (!a.use_graph) {
    for (int i = 0; i < a.nsteps; ++i) {
      if (int e = step(rs, t_dev, st, &d.launches)) return e;
      if (int e = advance_step_enqueue(d.d_step, t_dev, d.d_tsteps, a.nsteps, st)) return e;
      ++d.launches;
    }
  } else {
    const cm_chain_args& k = d.graph_key;
    const bool reuse = d.graph_exec && k.n == a.n && k.mode == a.mode && k.noise == a.noise &&
                       k.history == a.history && k.nsteps == a.nsteps && k.use_graph == a.use_graph;
    if (!reuse) {
      chain_drop_graph(d);
      if (int e = capture(d, a, rs, step)) return e;
    }
    d.graph_launches = a.use_graph == 1 ? a.nsteps : 1;
    for (int64_t i = 0; i < d.graph_launches; ++i) CM_CUDA(cudaGraphLaunch(d.graph_exec, st));
    d.launches = d.graph_launches_per_step * a.nsteps;
  }
  CM_CUDA(cudaMemcpyAsync(a.x, x_stage, x_bytes, cudaMemcpyDeviceToDevice, st));
  return 0;
}

}  // namespace cm
