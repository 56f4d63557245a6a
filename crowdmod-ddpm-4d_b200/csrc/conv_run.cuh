// Which kernel runs a conv: the one place that chooses among the forward conv kernels (conv_res32, conv_plane,
// conv_umma) and between the two weight-gradient schemes (wgrad_plane chunks, wgrad_umma).
#pragma once
#include <variant>

#include "conv_plane.cuh"
#include "conv_res32.cuh"
#include "conv_umma.cuh"
#include "kernels.cuh"
#include "wgrad_plane.cuh"
#include "wgrad_umma.cuh"

namespace cm {

enum ConvKind : unsigned { CONV_UMMA = 1, CONV_PLANE = 2, CONV_RES32 = 4 };

// One prepared launch of the kernel conv_run_prepare picked (std::monostate: none covers the conv)
struct ConvRun {
  std::variant<std::monostate, ConvLaunch, PlaneLaunch, Res32Launch> l;
  bool covered() const { return l.index() != 0; }
};

// Prepares the first of res32, plane, umma that `kinds` allows and that covers the conv (res32 and plane: mode 0 only),
// with epilogue `epi`.  Returns 0 with R not covered when none does (only possible without CONV_UMMA).
int conv_run_prepare(ConvRun* R, unsigned kinds, int mode, const __half* act, int B, int D, int H, int W, int cin,
                     const __half* extra, int cin_extra, const __half* wpacked, int cout, int terms,
                     const ConvEpilogue& epi);
int conv_run_enqueue(const ConvRun& R, cudaStream_t st);
ConvEpilogue& conv_run_epi(ConvRun& R);   // R must be covered
GnRec conv_run_records(const ConvRun& R);  // GroupNorm records the launch writes (units == 0: none)

// Weight gradient of one conv: plane / halo chunks (k3 s1 convs with 32 output channels: one launch per 32-channel
// chunk of the main source, the fused 1x1x1 source through wgrad_umma in 1x1x1 mode) or one wgrad_umma launch
struct WgradRun {
  WgradPlaneLaunch plane[8];
  int n_plane = 0;
  WgradLaunch umma;        // n_plane == 0: the whole gradient, else the rows of the 1x1x1 source
  bool has_umma = false;
  int launches() const { return n_plane + (has_umma ? 1 : 0); }
};

// Plane chunks when CONV_PLANE is allowed and covers the conv (up to 4 chunks next to CONV_UMMA, 8 alone), else umma
// when allowed; launches() == 0: not covered.  act_ld / dout_ld / extra_ld: row strides (0 = channel count).
int wgrad_run_prepare(WgradRun* R, unsigned kinds, int mode, const __half* act, int B, int D, int H, int W, int cin,
                      const __half* extra, int cin_extra, const __half* dout, int cout, float* G, int dout_ld = 0,
                      int act_ld = 0, int extra_ld = 0);
// part != nullptr: the deterministic variant (per-CTA / per-split partials in part, summed in a fixed order into G;
// two launches per kernel launch); part holds wgrad_run_partial_elems(R) floats.
int wgrad_run_enqueue(const WgradRun& R, cudaStream_t st, float* part = nullptr);
size_t wgrad_run_partial_elems(const WgradRun& R);

// Which kernels may take the weight gradient of the first conv (c = its cout) or the final conv (c = its cin) as a conv
// weight gradient over the packed fp16 operands (wgrad_run).  0: the SIMT kernels of backward.cu, which cover 32 and 64
// channels; 64 keeps them, 32 takes the plane kernel, wider layers the plane chunks or wgrad_umma.
inline unsigned edge_wgrad_kinds(int c) { return c == 32 ? CONV_PLANE : c == 64 ? 0u : CONV_UMMA | CONV_PLANE; }

}  // namespace cm
