// Host side of the tcgen05 implicit-GEMM conv: tensor-map construction and launch.
#include "conv_run.cuh"

#include <cudaTypedefs.h>
#include <string.h>

namespace cm {

namespace {

PFN_cuTensorMapEncodeTiled_v12000 g_encode_tiled = nullptr;
PFN_cuTensorMapEncodeIm2col_v12000 g_encode_im2col = nullptr;
int g_driver_version = 0;

int load_driver_syms() {
  if (g_encode_tiled && g_encode_im2col) return 0;
  cudaDriverEntryPointQueryResult q;
  void* fn = nullptr;
  CM_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
  CM_CHECK(fn != nullptr && q == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled not found");
  g_encode_tiled = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
  fn = nullptr;
  CM_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &fn, cudaEnableDefault, &q));
  CM_CHECK(fn != nullptr && q == cudaDriverEntryPointSuccess, "cuTensorMapEncodeIm2col not found");
  g_encode_im2col = reinterpret_cast<PFN_cuTensorMapEncodeIm2col_v12000>(fn);
  CM_CUDA(cudaDriverGetVersion(&g_driver_version));
  return 0;
}

}  // namespace

// Activation tensor [B, D, H, W, C] fp16 -> 5-D im2col map, dims ordered (C, W, H, D, N).
int make_act_map(CUtensorMap* map, const __half* base, int B, int D, int H, int W, int C, int bk,
                 int lower_w, int lower_h, int lower_d, int stride, int upper_delta, int ld) {
  // ld = channel stride of a pixel row in elements (0 -> C); ld > C views the first C channels of wider rows
  // (the hi half of a K-concatenated hi|lo dOut pair)
  const cuuint64_t Cs = (cuuint64_t)(ld > 0 ? ld : C);
  cuuint64_t dims[5] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)B};
  cuuint64_t strides[4] = {Cs * 2, (cuuint64_t)W * Cs * 2, (cuuint64_t)H * W * Cs * 2,
                           (cuuint64_t)D * H * W * Cs * 2};
  // For the forward conv shapes (k3 p1 s1|s2, 2x2x2 phase taps, 1x1x1) the upper corner
  // (upper_pad - (k-1)) equals the lower corner (-lower_pad); the k4 s2 dgrad of UpSample needs
  // upper = lower - 1 (upper_delta = -1).
  int lower[3] = {lower_w, lower_h, lower_d};
  int upper[3] = {lower_w + upper_delta, lower_h + upper_delta, lower_d + upper_delta};
  cuuint32_t estr[5] = {1, (cuuint32_t)stride, (cuuint32_t)stride, (cuuint32_t)stride, 1};
  CUtensorMapSwizzle sw = (bk == 64) ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  CUresult r = g_encode_im2col(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, (void*)base, dims, strides,
                               lower, upper, (cuuint32_t)bk, (cuuint32_t)CONV_BM, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  CM_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeIm2col failed: %d (B=%d D=%d H=%d W=%d C=%d bk=%d)",
           (int)r, B, D, H, W, C, bk);
  // Driver quirk mirrored from CUTLASS (cute/atom/copy_traits_sm90_im2col.hpp): for tensors
  // smaller than 128 KiB, drivers <= 13.1 set a descriptor bit that must be cleared.
  if (g_driver_version <= 13010) {
    size_t bytes = (size_t)B * D * H * W * Cs * 2;
    if (bytes < 131072) reinterpret_cast<uint64_t*>(map)[1] &= ~(1ull << 21);
  }
  return 0;
}

namespace {

int make_weight_map(CUtensorMap* map, const __half* base, size_t rows, size_t ktot, int bk, int bn) {
  cuuint64_t dims[2] = {(cuuint64_t)ktot, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ktot * 2};
  cuuint32_t box[2] = {(cuuint32_t)bk, (cuuint32_t)bn};
  cuuint32_t estr[2] = {1, 1};
  CUtensorMapSwizzle sw = (bk == 64) ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  CUresult r = g_encode_tiled(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, (void*)base, dims, strides,
                              box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  CM_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed: %d (rows=%zu k=%zu)", (int)r, rows,
           ktot);
  return 0;
}

template <int BN, int BK>
int launch_t(const ConvLaunch& L, cudaStream_t st) {
  if (L.p.ksplit > 1) {
    // the ksplit CTAs along z that share an output tile form one thread-block cluster
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = L.grid;
    cfg.blockDim = dim3(CONV_THREADS);
    cfg.dynamicSmemBytes = L.smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 1;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = L.p.ksplit;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (L.p.terms == 2) CM_CUDA(cudaLaunchKernelEx(&cfg, conv_umma_kernel<BN, BK, 2>, L.p));
    else CM_CUDA(cudaLaunchKernelEx(&cfg, conv_umma_kernel<BN, BK, 1>, L.p));
    return 0;
  }
  if (L.p.terms == 2) conv_umma_kernel<BN, BK, 2><<<L.grid, CONV_THREADS, L.smem, st>>>(L.p);
  else conv_umma_kernel<BN, BK, 1><<<L.grid, CONV_THREADS, L.smem, st>>>(L.p);
  CM_CUDA(cudaGetLastError());
  return 0;
}

template <int BN, int BK>
int set_attr_t() {
  CM_CUDA(cudaFuncSetAttribute(conv_umma_kernel<BN, BK, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               227 * 1024));
  CM_CUDA(cudaFuncSetAttribute(conv_umma_kernel<BN, BK, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               227 * 1024));
  return 0;
}

}  // namespace

int conv_init() {
  static bool done = false;
  if (done) return 0;
  if (int rc = load_driver_syms()) return rc;
  if (int rc = plane_init()) return rc;
  if (int rc = set_attr_t<128, 64>()) return rc;
  if (int rc = set_attr_t<64, 64>()) return rc;
  if (int rc = set_attr_t<32, 64>()) return rc;
  if (int rc = set_attr_t<128, 32>()) return rc;
  if (int rc = set_attr_t<64, 32>()) return rc;
  if (int rc = set_attr_t<32, 32>()) return rc;
  done = true;
  return 0;
}

size_t conv_packed_k(int mode, int cin, int cin_extra) {
  switch (mode) {
    case 0:
    case 1: return (size_t)27 * cin + cin_extra;
    case 2:
    case 4: return (size_t)64 * cin;
    default: return (size_t)cin + cin_extra;
  }
}

int conv_prepare(ConvLaunch* L, int mode, const __half* act, int B, int D, int H, int W, int cin,
                 const __half* extra, int cin_extra, const __half* wpacked, int cout, int terms, const ConvEpilogue& epi,
                 bool allow_splitk) {
  if (int rc = load_driver_syms()) return rc;
  CM_CHECK(mode >= 0 && mode <= 4, "bad conv mode %d", mode);
  CM_CHECK(cin % 32 == 0 && cin_extra % 32 == 0, "channels must be multiples of 32 (cin=%d extra=%d)",
           cin, cin_extra);
  CM_CHECK(cout % 32 == 0, "cout must be a multiple of 32 (%d)", cout);
  CM_CHECK(terms == 1 || terms == 2, "terms must be 1 or 2");
  CM_CHECK(!(mode == 2 && cin_extra), "upsample conv takes no extra source");
  memset(L, 0, sizeof(*L));
  ConvParams& p = L->p;
  const int bk = (cin % 64 == 0 && cin_extra % 64 == 0) ? 64 : 32;
  int stride = 1, k = 3, od = D, oh = H, ow = W;
  if (mode == 1) {
    stride = 2;
    od = (D - 1) / 2 + 1;
    oh = (H - 1) / 2 + 1;
    ow = (W - 1) / 2 + 1;
  } else if (mode == 2) {
    k = 2;
  } else if (mode == 3) {
    k = 1;
  } else if (mode == 4) {   // k4 s2, pad (1,2): data gradient of nearest-x2 + k3 (UpSample)
    stride = 2;
    k = 4;
    od = D / 2;
    oh = H / 2;
    ow = W / 2;
  }
  p.nphase = (mode == 2) ? 8 : 1;
  // N tile: as wide as possible (A is re-read once per N tile) unless that leaves most SMs idle
  // (coarse levels have only a few dozen M tiles): then trade A re-reads for more CTAs.
  int bn = (cout % 128 == 0) ? 128 : (cout % 64 == 0 ? 64 : 32);
  int ksplit = 1;
  {
    const long m_tiles = ((long)B * od * oh * ow + CONV_BM - 1) / CONV_BM * p.nphase;
    // M-starved deep-K layers (coarsest level: a few dozen M tiles, K in the thousands): keep the
    // widest N tile (A and the weights are fetched once per tile) and split K across a cluster.
    const long nkb_all = (long)(k * k * k) * (cin / bk) + cin_extra / bk;
    if (allow_splitk && p.nphase == 1 && m_tiles * (cout / bn) < 100) {
      long sk = 2 * 148 / (m_tiles * (cout / bn));   // two CTAs per SM (see the stage budget below)
      if (sk > 8) sk = 8;
      while (sk > 1 && nkb_all / sk < 4) --sk;
      if (sk >= 2) ksplit = (int)sk;
    }
    if (ksplit == 1)
      while (bn > 32 && m_tiles * (cout / bn) < 120) bn >>= 1;
  }
  L->bk = bk;
  L->bn = bn;
  for (int ph = 0; ph < p.nphase; ++ph) {
    int lw, lh, ld;
    if (mode == 2) {
      lw = (ph & 1) ? 0 : -1;
      lh = (ph & 2) ? 0 : -1;
      ld = (ph & 4) ? 0 : -1;
    } else if (mode == 3) {
      lw = lh = ld = 0;
    } else {
      lw = lh = ld = -1;
    }
    p.lower[ph][0] = (signed char)lw;
    p.lower[ph][1] = (signed char)lh;
    p.lower[ph][2] = (signed char)ld;
    if (int rc = make_act_map(&p.amap[ph], act, B, D, H, W, cin, bk, lw, lh, ld, stride, mode == 4 ? -1 : 0)) return rc;
  }
  if (cin_extra) {
    CM_CHECK(extra != nullptr, "extra source pointer missing");
    if (int rc = make_act_map(&p.xmap, extra, B, od, oh, ow, cin_extra, bk, 0, 0, 0, 1, 0)) return rc;
  }
  const size_t ktot = conv_packed_k(mode, cin, cin_extra);
  if (int rc = make_weight_map(&p.bmap, wpacked, (size_t)terms * cout, ktot, bk, bn)) return rc;

  p.M = B * od * oh * ow;
  p.od = od;
  p.oh = oh;
  p.ow = ow;
  p.pps = od * oh * ow;
  p.conv_stride = stride;
  p.kd = p.kh = p.kw = k;
  p.cin_main = cin;
  p.cin_extra = cin_extra;
  p.kphase = (mode == 2) ? 8 * cin : 0;
  p.terms = terms;
  p.cout = cout;
  p.epi = epi;
  p.epi.stats_rec = nullptr;   // a request: this kernel writes no GroupNorm records
  p.epi.out_ld = cout;
  p.scatter = (mode == 2) ? 1 : 0;
  p.err_flag = device_error_flag();

  const int stage_bytes = CONV_BM * bk * 2 + terms * bn * bk * 2;
  // Few CTAs (coarse levels: 27 M tiles) are TMA-latency bound: give each all the shared memory
  // it can use.  Many CTAs per SM: keep stages modest so that several CTAs stay co-resident.
  int stages = 4;
  {
    const long ctas = (long)((p.M + CONV_BM - 1) / CONV_BM) * (cout / bn) * p.nphase;
    const long per_sm = (ctas + 147) / 148;
    const long budget = 200 * 1024 / (per_sm < 3 ? per_sm : 3);
    const long fit = budget / stage_bytes;
    if (fit > stages) stages = (int)(fit < CONV_MAX_STAGES ? fit : CONV_MAX_STAGES);
  }
  // UpSample phase convs have only 8 k-blocks per phase: co-residency (>= 3 CTAs per SM hiding each
  // other's set-up and epilogue) beats pipeline depth (measured: 51.6 us with 2 stages vs 63.7 with 4)
  if (p.nphase == 8) stages = 2;
  if (stages > CONV_MAX_STAGES) stages = CONV_MAX_STAGES;
  while (stages > 2 && (size_t)stages * stage_bytes + 2048 > 200 * 1024) --stages;
  p.stages = stages;
  p.ksplit = 1;
  if (ksplit > 1) {
    const int nkb_all = k * k * k * (cin / bk) + cin_extra / bk;
    p.kb_per_split = (nkb_all + ksplit - 1) / ksplit;
    ksplit = (nkb_all + p.kb_per_split - 1) / p.kb_per_split;          // no empty CTA
    // Two CTAs per SM (<= ~100 KB of stages each): a cluster must be co-scheduled inside one GPC, and
    // with one 200 KB CTA per SM the 27 x S CTAs of a coarse-level conv did not fit one wave (measured:
    // 2 waves of 9 us instead of 1).  The partial tile [128][bn + 4] fp32 is staged over the
    // pipeline buffers, which bounds the stage count from below.
    stages = (int)((100 * 1024) / stage_bytes);
    if (stages < 2) stages = 2;
    if (stages > CONV_MAX_STAGES) stages = CONV_MAX_STAGES;
    while ((size_t)stages * stage_bytes < (size_t)CONV_BM * (bn + 4) * 4 && stages < CONV_MAX_STAGES) ++stages;
    CM_CHECK((size_t)stages * stage_bytes >= (size_t)CONV_BM * (bn + 4) * 4, "split-K staging does not fit");
    p.stages = stages;
    p.ksplit = ksplit;
  }
  L->smem = (size_t)stages * stage_bytes + 1024 /*align slack*/ + 256 /*barriers*/ + 512 /*colv*/;
  // scatter convs: 4 phases per CTA when that still leaves >= 2 CTAs per SM, else 2, else 1
  p.ppc = 1;
  if (p.nphase == 8) {
    const long tiles = (long)((p.M + CONV_BM - 1) / CONV_BM) * (cout / bn);
    if (tiles * 2 >= 296) p.ppc = 4;
    else if (tiles * 4 >= 296) p.ppc = 2;
  }
  L->grid = dim3((p.M + CONV_BM - 1) / CONV_BM, cout / bn, p.ksplit > 1 ? p.ksplit : p.nphase / p.ppc);
  return 0;
}

int conv_enqueue(const ConvLaunch& L, cudaStream_t st) {
  if (L.bk == 64) {
    if (L.bn == 128) return launch_t<128, 64>(L, st);
    if (L.bn == 64) return launch_t<64, 64>(L, st);
    return launch_t<32, 64>(L, st);
  } else {
    if (L.bn == 128) return launch_t<128, 32>(L, st);
    if (L.bn == 64) return launch_t<64, 32>(L, st);
    return launch_t<32, 32>(L, st);
  }
}



// ================================ plane-tile conv (conv_plane.cuh) ================================
namespace {

// packed weights [rows][Ktot] viewed as (k within a tap slab, row, tap slab): box {bk, bn, 9} = the nine
// (th, tw) slabs of one td, laid out slab-major in shared memory ([slab][bn rows][bk])
int make_weight_map3(CUtensorMap* map, const __half* base, size_t rows, size_t ktot, int cin, int bk, int bn) {
  cuuint64_t dims[3] = {(cuuint64_t)cin, (cuuint64_t)rows, 27};
  cuuint64_t strides[2] = {(cuuint64_t)ktot * 2, (cuuint64_t)cin * 2};
  cuuint32_t box[3] = {(cuuint32_t)bk, (cuuint32_t)bn, 9};
  cuuint32_t estr[3] = {1, 1, 1};
  CUtensorMapSwizzle sw = (bk == 64) ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  CUresult r = g_encode_tiled(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, (void*)base, dims, strides, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  CM_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (3-D weights) failed: %d (rows=%zu k=%zu cin=%d)", (int)r, rows,
           ktot, cin);
  return 0;
}

int make_plane_map(CUtensorMap* map, const __half* base, int B, int D, int H, int W, int C, int bk, int R,
                   int HB) {
  cuuint64_t dims[5] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)B};
  cuuint64_t strides[4] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2,
                           (cuuint64_t)D * H * W * C * 2};
  cuuint32_t box[5] = {(cuuint32_t)bk, (cuuint32_t)(W + 2), (cuuint32_t)HB, (cuuint32_t)R, 1};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUtensorMapSwizzle sw = (bk == 64) ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  CUresult r = g_encode_tiled(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, (void*)base, dims, strides, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  CM_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (plane) failed: %d (B=%d D=%d H=%d W=%d C=%d R=%d)", (int)r,
           B, D, H, W, C, R);
  return 0;
}

template <int BN, int BK>
int plane_launch_t(const PlaneLaunch& L, cudaStream_t st) {
  if (L.p.terms == 2) conv_plane_kernel<BN, BK, 2><<<L.grid, PL_THREADS, L.smem, st>>>(L.p);
  else conv_plane_kernel<BN, BK, 1><<<L.grid, PL_THREADS, L.smem, st>>>(L.p);
  CM_CUDA(cudaGetLastError());
  return 0;
}
template <int BN, int BK>
int plane_attr_t() {
  CM_CUDA(cudaFuncSetAttribute(conv_plane_kernel<BN, BK, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  CM_CUDA(cudaFuncSetAttribute(conv_plane_kernel<BN, BK, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  return 0;
}

}  // namespace

int plane_init() {
  static bool done = false;
  if (done) return 0;
  if (int rc = load_driver_syms()) return rc;
  if (int rc = plane_attr_t<32, 32>()) return rc;
  if (int rc = plane_attr_t<32, 64>()) return rc;
  if (int rc = plane_attr_t<64, 32>()) return rc;
  if (int rc = plane_attr_t<64, 64>()) return rc;
  if (int rc = plane_attr_t<128, 32>()) return rc;
  if (int rc = plane_attr_t<128, 64>()) return rc;
  done = true;
  return 0;
}

int plane_prepare(PlaneLaunch* L, const __half* act, int B, int D, int H, int W, int cin,
                  const __half* extra, int cin_extra, const __half* wpacked, int cout, int terms, const ConvEpilogue& epi) {
  if (int rc = load_driver_syms()) return rc;
  memset(L, 0, sizeof(*L));
  L->ok = false;
  if (cin % 32 || cin_extra % 32 || cout % 32) return 0;
  const int Wp = W + 2;
  if (Wp > 256 || H > 256) return 0;
  static int n_sm = 0;
  if (!n_sm) {
    int dev = 0;
    CM_CUDA(cudaGetDevice(&dev));
    CM_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
  }
  int bk = (cin % 64 == 0 && cin_extra % 64 == 0) ? 64 : 32;
  int bn = (cout % 128 == 0) ? 128 : (cout % 64 == 0 ? 64 : 32);
  while (bn > 32 && 3 * bn > 256) bn >>= 1;             // tw-stacked MMA: N = 3*BN <= 256
  const int nst = 3 * bn;
  int rowb = bk * 2;
  const int max_tiles = 256 / nst;                      // two accumulator buffers in 512 TMEM columns
  if (max_tiles < 1) return 0;
  const long smem_cap = 220 * 1024;
  const long tail_fixed = 256 + 512 + 1024;
  auto ybuf_bytes = [&](int ntiles) {
    return (long)(ntiles * 128 + 2) * (bn + 4) * 4 + (long)(ntiles * 4 + 1) * 3 * bn * 4 + (long)((PL_EPI / 32) * bn * 2 + bn) * 4;
  };
  // work unit: R planes x HB rows.  Score = useful MMA rows x SM fill of the last wave; ties go to
  // the larger unit (more reuse of every weight tile).
  int bestR = 0, bestHB = 0;
  double best = 0.0;
  auto consider = [&](int R, int HB) {
    const int P = R * HB * Wp;
    const int ntiles = (P + 127) / 128;
    if (ntiles > max_tiles || R > 256 || HB > 256) return;
    if (ntiles * 128 > PL_NJ * (PL_EPI / (bn / 4))) return;    // PL_NJ store rows per epilogue thread
    const long a_stage = ((long)(ntiles * 128 + 8) * rowb + 1023) / 1024 * 1024;
    const long stage = a_stage + (long)terms * nst * rowb;
    if (2 * stage + tail_fixed + ybuf_bytes(ntiles) > smem_cap) return;
    const long units = (long)B * (D / R) * (H / HB) * (cout / bn);
    const long waves = (units + n_sm - 1) / n_sm;
    const double eff = (double)R * HB * W / (ntiles * 128.0);
    if (eff < 0.6) return;                               // mostly padding: leave it to conv_umma
    // useful rows per modelled CTA time: a unit costs its MMAs (~55 cycles each, tw taps stacked along N) plus a fixed
    // ~2 600 cycles and ~310 cycles per pipeline stage whatever it computes (knock-out skeleton runs, DESIGN.md 3.1.5:
    // 2.3 us per unit on the HERMES grid) -- fewer, fatter units win when the rows-per-tile efficiency is close.
    const double bk_model = R == 1 ? 32.0 : (double)bk;   // th3 stages (single-plane units) use BK = 32
    const double mma_tile = 55.0 * (9.0 * (cin / 16) + (cin_extra / 16)) * terms;
    const double stages = (R == 1 ? 3.0 : 9.0) * (cin / bk_model) + cin_extra / bk_model;
    const double unit_cost = 2600.0 + 310.0 * stages;
    const double score = eff * ((double)units / (waves * n_sm)) * (ntiles * mma_tile) / (ntiles * mma_tile + unit_cost);
    if (score > best * 1.0001 || (score > best * 0.9999 && R * HB > bestR * bestHB)) {
      best = score;
      bestR = R;
      bestHB = HB;
    }
  };
  for (int hb = 1; hb <= H; ++hb)
    if (H % hb == 0) consider(1, hb);
  for (int r = 2; r <= D; ++r)
    if (D % r == 0) consider(r, H);
  if (bestR == 0) return 0;
  const int R = bestR, HB = bestHB;
  const int P = R * HB * Wp;
  const int ntiles = (P + 127) / 128;
  PlaneParams& p = L->p;
  // th3 mode (see PlaneParams::th3): single-plane units only; BK = 32 keeps the nine-slab weight stage small
  bool th3 = R == 1;
  if (th3) {
    // needs two stages of {A halo box, nine weight slabs per term} next to the epilogue buffers
    const long a3 = ((long)(ntiles * 128 + 2 * Wp) * 64 + 1023) / 1024 * 1024;
    const long stage3 = a3 + (long)terms * 3 * nst * 64;
    if ((smem_cap - (tail_fixed + ybuf_bytes(ntiles))) / stage3 < 2) th3 = false;
  }
  if (th3) {
    bk = 32;
    rowb = bk * 2;
  }
  if (int rc = make_plane_map(&p.amap, act, B, D, H, W, cin, bk, R, th3 ? HB + 2 : HB)) return rc;
  if (cin_extra) {
    CM_CHECK(extra != nullptr, "extra source pointer missing");
    if (int rc = make_plane_map(&p.xmap, extra, B, D, H, W, cin_extra, bk, R, HB)) return rc;
  }
  const size_t ktot = conv_packed_k(0, cin, cin_extra);
  if (int rc = make_weight_map(&p.bmap, wpacked, (size_t)terms * cout, ktot, bk, bn)) return rc;
  if (th3)
    if (int rc = make_weight_map3(&p.bmap3, wpacked, (size_t)terms * cout, ktot, cin, bk, bn)) return rc;
  p.th3 = th3 ? 1 : 0;
  p.a_box_bytes = (th3 ? (HB + 2) * Wp : P) * rowb;
  p.H = H; p.W = W; p.D = D; p.Wp = Wp; p.R = R; p.HB = HB; p.P = P; p.ntiles = ntiles;
  p.units_per_sample = (D / R) * (H / HB);
  p.n_ntiles = cout / bn;
  p.n_units = B * p.units_per_sample * p.n_ntiles;
  p.a_stage_bytes = (int)(((long)(ntiles * 128 + (th3 ? 2 * Wp : 8)) * rowb + 1023) / 1024 * 1024);
  p.cin_main = cin; p.cin_extra = cin_extra; p.cout = cout; p.terms = terms;
  p.epi = epi;
  p.epi.out_ld = cout;
  p.err_flag = device_error_flag();
  const long stage = p.a_stage_bytes + (long)terms * (th3 ? 3 : 1) * nst * rowb;
  const long tail = tail_fixed + ybuf_bytes(ntiles);
  int stages = (int)((smem_cap - tail) / stage);
  if (stages > PL_MAX_STAGES) stages = PL_MAX_STAGES;
  if (stages < 2) return 0;
  p.stages = stages;
  L->bn = bn;
  L->bk = bk;
  L->smem = (size_t)stages * stage + tail;
  L->grid = dim3(p.n_units < n_sm ? p.n_units : n_sm, 1, 1);
  L->ok = true;
  return 0;
}

int plane_enqueue(const PlaneLaunch& L, cudaStream_t st) {
  if (L.bk == 64) {
    if (L.bn == 128) return plane_launch_t<128, 64>(L, st);
    if (L.bn == 64) return plane_launch_t<64, 64>(L, st);
    return plane_launch_t<32, 64>(L, st);
  }
  if (L.bn == 128) return plane_launch_t<128, 32>(L, st);
  if (L.bn == 64) return plane_launch_t<64, 32>(L, st);
  return plane_launch_t<32, 32>(L, st);
}

// ================================ weights-resident 32 -> 32 conv (conv_res32.cuh) ================================
int res32_init() {
  static bool done = false;
  if (done) return 0;
  if (int rc = load_driver_syms()) return rc;
  CM_CUDA(cudaFuncSetAttribute(conv_res32_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  done = true;
  return 0;
}

int res32_prepare(Res32Launch* L, const __half* act, int B, int D, int H, int W, int cin, const __half* extra,
                  int cin_extra, const __half* wpacked, int cout, int terms, const ConvEpilogue& epi) {
  if (int rc = res32_init()) return rc;
  memset(L, 0, sizeof(*L));
  L->ok = false;
  if (cin != R32_C || cout != R32_C || terms != 2 || cin_extra % R32_C || cin_extra > 3 * R32_C) return 0;
  const int Wp = W + 2;
  if (Wp > 128 || H > 256) return 0;   // H: conv_plane's limit; res32 stands in for conv_plane, never for conv_umma alone
  int HB = 0;
  for (int hb = 1; hb <= H; ++hb)
    if (H % hb == 0 && hb * Wp <= 128) HB = hb;
  if (HB == 0 || HB + 2 > 256 || (double)HB * W / 128.0 < 0.6) return 0;
  static int n_sm = 0;
  if (!n_sm) {
    int dev = 0;
    CM_CUDA(cudaGetDevice(&dev));
    CM_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
  }
  Res32Params& p = L->p;
  const int nx = cin_extra / R32_C;
  // a stage holds one haloed plane box; the th = 2 view of a 128-row MMA reads up to row 2*Wp + 127
  const int stage_bytes = (int)(((long)(2 * Wp + 128) * 64 + 1023) / 1024 * 1024);
  const long tail = 256 + 2 * R32_C * 4 + 2 * 8 * R32_C * 2 * 4 + 2 * 5 * 3 * R32_C * 4 + 2L * 128 * R32_TLD * 4;
  const long fixed = 9L * R32_WBLK + (long)nx * R32_WX + tail + 1024;
  int stages = (int)((227L * 1024 - fixed) / stage_bytes);
  if (stages > R32_MAX_STAGES) stages = R32_MAX_STAGES;
  if (stages < 3) return 0;
  CM_CHECK(epi.lo_from == 0 && epi.lo_from_x == 0 && epi.out16_lo == 0,
           "weights-resident conv: hi|lo operand pairs are not supported");
  CM_CHECK(epi.out16_ld == 0 || epi.out16_ld == R32_C, "weights-resident conv: fp16 rows of %d channels", epi.out16_ld);
  if (int rc = make_plane_map(&p.amap, act, B, D, H, W, R32_C, 32, 1, HB + 2)) return rc;
  if (nx) {
    CM_CHECK(extra != nullptr, "extra source pointer missing");
    if (int rc = make_plane_map(&p.xmap, extra, B, D, H, W, cin_extra, 32, 1, HB)) return rc;
  }
  const size_t ktot = conv_packed_k(0, cin, cin_extra);
  {
    // packed weights [2*32 rows][Ktot] viewed as (k within a tap slab, row, tap slab): box {32, 64, 3} = the
    // three tw slabs of one (td, th), hi rows then lo rows -> [tw][hi|lo][co] rows of 64 B in shared memory
    cuuint64_t dims[3] = {(cuuint64_t)R32_C, (cuuint64_t)(2 * R32_C), 27};
    cuuint64_t strides[2] = {(cuuint64_t)ktot * 2, (cuuint64_t)R32_C * 2};
    cuuint32_t box[3] = {(cuuint32_t)R32_C, (cuuint32_t)(2 * R32_C), 3};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = g_encode_tiled(&p.wmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, (void*)wpacked, dims, strides, box, estr,
                                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B,
                                CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    CM_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (resident weights) failed: %d (k=%zu)", (int)r, ktot);
  }
  if (nx)
    if (int rc = make_weight_map(&p.wxmap, wpacked, (size_t)2 * R32_C, ktot, 32, 2 * R32_C)) return rc;
  p.H = H; p.W = W; p.D = D; p.Wp = Wp; p.HB = HB; p.P = HB * Wp;
  p.units_per_sample = D * (H / HB);
  p.n_units = B * p.units_per_sample;
  p.nx = nx;
  p.stages = stages;
  p.stage_bytes = stage_bytes;
  p.epi = epi;
  p.epi.out_ld = R32_C;
  p.err_flag = device_error_flag();
  L->smem = (size_t)fixed + (size_t)stages * stage_bytes;
  L->grid = dim3(p.n_units < n_sm ? p.n_units : n_sm, 1, 1);
  L->ok = true;
  return 0;
}

int res32_enqueue(const Res32Launch& L, cudaStream_t st) {
  conv_res32_kernel<2><<<L.grid, R32_THREADS, L.smem, st>>>(L.p);
  CM_CUDA(cudaGetLastError());
  return 0;
}

// ================================ weight gradient (wgrad_umma.cuh) ================================
namespace {

template <int BKC, int BNC, int BN>
int wg_launch_t(const WgradLaunch& L, cudaStream_t st) {
  wgrad_umma_kernel<BKC, BNC, BN><<<L.grid, WG_THREADS, L.smem, st>>>(L.p);
  CM_CUDA(cudaGetLastError());
  return 0;
}
template <int BKC, int BNC, int BN>
int wg_attr_t() {
  CM_CUDA(cudaFuncSetAttribute(wgrad_umma_kernel<BKC, BNC, BN>,
                               cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  return 0;
}
template <int BKC>
int wg_dispatch(const WgradLaunch& L, cudaStream_t st) {
  if (L.bnc == 32) return wg_launch_t<BKC, 32, 32>(L, st);
  switch (L.bn) {
    case 64: return wg_launch_t<BKC, 64, 64>(L, st);
    case 128: return wg_launch_t<BKC, 64, 128>(L, st);
    default: return wg_launch_t<BKC, 64, 256>(L, st);
  }
}

}  // namespace

int wgrad_init() {
  static bool done = false;
  if (done) return 0;
  if (int rc = load_driver_syms()) return rc;
  if (int rc = wgrad_plane_init()) return rc;
  if (int rc = wg_attr_t<32, 32, 32>()) return rc;
  if (int rc = wg_attr_t<32, 64, 64>()) return rc;
  if (int rc = wg_attr_t<32, 64, 128>()) return rc;
  if (int rc = wg_attr_t<32, 64, 256>()) return rc;
  if (int rc = wg_attr_t<64, 32, 32>()) return rc;
  if (int rc = wg_attr_t<64, 64, 64>()) return rc;
  if (int rc = wg_attr_t<64, 64, 128>()) return rc;
  if (int rc = wg_attr_t<64, 64, 256>()) return rc;
  done = true;
  return 0;
}

size_t wgrad_g_elems(int mode, int cin, int cin_extra, int cout) {
  return conv_packed_k(mode, cin, cin_extra) * (size_t)cout;
}

int wgrad_prepare(WgradLaunch* L, int mode, const __half* act, int B, int D, int H, int W, int cin,
                  const __half* extra, int cin_extra, const __half* dout, int cout, float* G, int dout_ld,
                  int act_ld, int extra_ld) {
  if (int rc = load_driver_syms()) return rc;
  CM_CHECK(mode >= 0 && mode <= 3, "bad wgrad mode %d", mode);
  CM_CHECK(cin % 32 == 0 && cin_extra % 32 == 0 && cout % 32 == 0,
           "channels must be multiples of 32 (cin=%d extra=%d cout=%d)", cin, cin_extra, cout);
  CM_CHECK(!(mode == 2 && cin_extra), "upsample conv takes no extra source");
  memset(L, 0, sizeof(*L));
  WgradParams& p = L->p;
  const int bkc = (cin % 64 == 0 && cin_extra % 64 == 0) ? 64 : 32;
  const int bnc = (cout % 64 == 0) ? 64 : 32;
  int bn = 32;
  if (bnc == 64) bn = (cout % 256 == 0) ? 256 : (cout % 128 == 0 ? 128 : 64);
  int stride = 1, k = 3, od = D, oh = H, ow = W;
  if (mode == 1) {
    stride = 2;
    od = (D - 1) / 2 + 1;
    oh = (H - 1) / 2 + 1;
    ow = (W - 1) / 2 + 1;
  } else if (mode == 2) {
    k = 2;
  } else if (mode == 3) {
    k = 1;
  }
  p.nphase = (mode == 2) ? 8 : 1;
  p.gstride = (mode == 2) ? 2 : 1;
  for (int ph = 0; ph < p.nphase; ++ph) {
    int lw = -1, lh = -1, ld = -1;
    if (mode == 2) {
      lw = (ph & 1) ? 0 : -1;
      lh = (ph & 2) ? 0 : -1;
      ld = (ph & 4) ? 0 : -1;
    } else if (mode == 3) {
      lw = lh = ld = 0;
    }
    p.lower[ph][0] = (signed char)lw;
    p.lower[ph][1] = (signed char)lh;
    p.lower[ph][2] = (signed char)ld;
    if (int rc = make_act_map(&p.amap[ph], act, B, D, H, W, cin, bkc, lw, lh, ld, stride, 0, act_ld)) return rc;
    if (mode == 2) {
      // dOut lives on the 2x grid; phase ph owns the pixels (2z+pz, 2p+pp, 2q+pq)
      const int gw = ph & 1, gh = (ph >> 1) & 1, gd = (ph >> 2) & 1;
      p.glower[ph][0] = (signed char)gw;
      p.glower[ph][1] = (signed char)gh;
      p.glower[ph][2] = (signed char)gd;
      if (int rc = make_act_map(&p.gmap[ph], dout, B, 2 * D, 2 * H, 2 * W, cout, bnc, gw, gh, gd, 2, -1, dout_ld))
        return rc;
    } else {
      if (int rc = make_act_map(&p.gmap[ph], dout, B, od, oh, ow, cout, bnc, 0, 0, 0, 1, 0, dout_ld)) return rc;
    }
  }
  if (cin_extra) {
    CM_CHECK(extra != nullptr, "extra source pointer missing");
    if (int rc = make_act_map(&p.xmap, extra, B, od, oh, ow, cin_extra, bkc, 0, 0, 0, 1, 0, extra_ld)) return rc;
  }
  p.M = B * od * oh * ow;
  p.od = od;
  p.oh = oh;
  p.ow = ow;
  p.pps = od * oh * ow;
  p.conv_stride = stride;
  p.kd = p.kh = p.kw = k;
  p.cin_main = cin;
  p.cin_extra = cin_extra;
  p.cout = cout;
  p.ncm = cin / bkc;
  p.atoms_main = k * k * k * p.ncm;
  p.atoms_total = p.atoms_main + cin_extra / bkc;
  p.apt = 128 / bkc;
  p.n_tiles = cout / bn;
  p.kb_total = (p.M + WG_KT - 1) / WG_KT;
  p.krows = k * k * k * cin + cin_extra;
  p.G = G;
  p.err_flag = device_error_flag();
  const int m_tiles = (p.atoms_total + p.apt - 1) / p.apt;
  // split the pixel reduction so that ~2 waves of CTAs cover the 148 SMs
  int splits = (2 * 148) / (m_tiles * p.n_tiles * p.nphase);
  if (splits < 1) splits = 1;
  if (splits > p.kb_total) splits = p.kb_total;
  p.kb_per_split = (p.kb_total + splits - 1) / splits;
  splits = (p.kb_total + p.kb_per_split - 1) / p.kb_per_split;   // no empty CTA
  p.splits = splits;
  const int stage_bytes = 128 * WG_KT * 2 + bn * WG_KT * 2;
  int stages = WG_MAX_STAGES;
  while (stages > 2 && (size_t)stages * stage_bytes + 2048 > 200 * 1024) --stages;
  p.stages = stages;
  L->bkc = bkc;
  L->bnc = bnc;
  L->bn = bn;
  L->smem = (size_t)stages * stage_bytes + 1024 + 256;
  L->grid = dim3(m_tiles, p.n_tiles * splits, p.nphase);
  return 0;
}

// ================================ weight gradient, plane / halo scheme (wgrad_plane.cuh) ================================
namespace {
int make_plane_box_map(CUtensorMap* map, const __half* base, int B, int D, int H, int W, int C, int ld, int box_w, int box_h) {
  cuuint64_t dims[5] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)B};
  cuuint64_t strides[4] = {(cuuint64_t)ld * 2, (cuuint64_t)W * ld * 2, (cuuint64_t)H * W * ld * 2,
                           (cuuint64_t)D * H * W * ld * 2};
  cuuint32_t box[5] = {32, (cuuint32_t)box_w, (cuuint32_t)box_h, 1, 1};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = g_encode_tiled(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, (void*)base, dims, strides, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  CM_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (wgrad plane box) failed: %d (B=%d D=%d H=%d W=%d C=%d ld=%d box %dx%d)",
           (int)r, B, D, H, W, C, ld, box_w, box_h);
  return 0;
}
}  // namespace

int wgrad_plane_prepare(WgradPlaneLaunch* L, const __half* act, int B, int D, int H, int W, int cin, int act_ld, int c0,
                        const __half* dout, int dout_ld, int cout, float* G) {
  if (int rc = load_driver_syms()) return rc;
  memset(L, 0, sizeof(*L));
  L->ok = false;
  if (cout != 32 || cin % 32 != 0 || c0 % 32 != 0 || c0 + 32 > cin) return 0;
  const int Wp = W + 2;
  const int HB = (Wp % 2 == 0) ? 6 : 14;                     // (HB + 2) * Wp must be a multiple of 16 (pixels per MMA)
  if (Wp > 256 || HB + 3 > 256 || ((HB + 2) * Wp) % 16 != 0) return 0;
  if (act_ld <= 0) act_ld = cin;
  if (dout_ld <= 0) dout_ld = cout;
  WgradPlaneParams& p = L->p;
  p.H = H; p.W = W; p.D = D; p.Wp = Wp; p.HB = HB;
  p.hblocks = (H + HB - 1) / HB;
  p.units_per_sample = D * p.hblocks;
  p.n_units = B * p.units_per_sample;
  p.c0 = c0;
  p.ksteps = (HB + 2) * Wp / 16;
  p.a_box_bytes = (HB + 3) * Wp * 64;
  p.a_slot_bytes = (p.a_box_bytes + 1023) & ~1023;
  p.g_box_bytes = HB * Wp * 64;
  p.g_data_off = (2 * Wp * 64 + 1023) & ~1023;               // zero guard rows in front of the box (>= two grid rows)
  p.g_slot_bytes = (p.g_data_off + p.g_box_bytes + 2 * Wp * 64 + 1023) & ~1023;
  p.stage_bytes = 3 * p.a_slot_bytes + p.g_slot_bytes;
  int stages = (int)((227L * 1024 - 1024 - 256) / p.stage_bytes);
  if (stages > WP_MAX_STAGES) stages = WP_MAX_STAGES;
  if (stages < 2) return 0;
  p.stages = stages;
  p.cin = cin;
  p.G = G;
  p.err_flag = device_error_flag();
  if (int rc = make_plane_box_map(&p.amap, act, B, D, H, W, cin, act_ld, Wp, HB + 3)) return rc;
  if (int rc = make_plane_box_map(&p.gmap, dout, B, D, H, W, cout, dout_ld, Wp, HB)) return rc;
  int n_sm = 148;
  cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, 0);
  L->grid = dim3(p.n_units < n_sm ? p.n_units : n_sm, 1, 1);
  L->smem = (size_t)stages * p.stage_bytes + 1024 + 256;
  L->ok = true;
  return 0;
}

int wgrad_plane_enqueue(const WgradPlaneLaunch& L, cudaStream_t st) {
  wgrad_plane_kernel<32><<<L.grid, WP_THREADS, L.smem, st>>>(L.p);
  CM_CUDA(cudaGetLastError());
  return 0;
}

int wgrad_plane_init() {
  static bool done = false;
  if (done) return 0;
  CM_CUDA(cudaFuncSetAttribute(wgrad_plane_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  done = true;
  return 0;
}

int wgrad_enqueue(const WgradLaunch& L, cudaStream_t st) {
  if (L.bkc == 64) return wg_dispatch<64>(L, st);
  return wg_dispatch<32>(L, st);
}

// ================================ kernel choice (conv_run.cuh) ================================
int conv_run_prepare(ConvRun* R, unsigned kinds, int mode, const __half* act, int B, int D, int H, int W, int cin,
                     const __half* extra, int cin_extra, const __half* wpacked, int cout, int terms,
                     const ConvEpilogue& epi) {
  if (mode == 0 && (kinds & CONV_RES32)) {
    Res32Launch& L = R->l.emplace<Res32Launch>();
    if (int rc = res32_prepare(&L, act, B, D, H, W, cin, extra, cin_extra, wpacked, cout, terms, epi)) return rc;
    if (L.ok) return 0;
  }
  if (mode == 0 && (kinds & CONV_PLANE)) {
    PlaneLaunch& L = R->l.emplace<PlaneLaunch>();
    if (int rc = plane_prepare(&L, act, B, D, H, W, cin, extra, cin_extra, wpacked, cout, terms, epi)) return rc;
    if (L.ok) return 0;
  }
  R->l = std::monostate{};
  if (kinds & CONV_UMMA)
    return conv_prepare(&R->l.emplace<ConvLaunch>(), mode, act, B, D, H, W, cin, extra, cin_extra, wpacked, cout, terms, epi);
  return 0;
}

int conv_run_enqueue(const ConvRun& R, cudaStream_t st) {
  if (const auto* L = std::get_if<Res32Launch>(&R.l)) return res32_enqueue(*L, st);
  if (const auto* L = std::get_if<PlaneLaunch>(&R.l)) return plane_enqueue(*L, st);
  CM_CHECK(R.covered(), "conv launch not prepared");
  return conv_enqueue(std::get<ConvLaunch>(R.l), st);
}

ConvEpilogue& conv_run_epi(ConvRun& R) {
  if (auto* L = std::get_if<Res32Launch>(&R.l)) return L->p.epi;
  if (auto* L = std::get_if<PlaneLaunch>(&R.l)) return L->p.epi;
  return std::get<ConvLaunch>(R.l).p.epi;
}

GnRec conv_run_records(const ConvRun& R) {
  if (const auto* L = std::get_if<Res32Launch>(&R.l))
    if (L->p.epi.stats_rec) return GnRec{L->p.epi.stats_rec, L->p.units_per_sample, L->p.HB * L->p.W};
  if (const auto* L = std::get_if<PlaneLaunch>(&R.l))
    if (L->p.epi.stats_rec) return GnRec{L->p.epi.stats_rec, L->p.units_per_sample, L->p.R * L->p.HB * L->p.W};
  return GnRec{};
}

int wgrad_run_prepare(WgradRun* R, unsigned kinds, int mode, const __half* act, int B, int D, int H, int W, int cin,
                      const __half* extra, int cin_extra, const __half* dout, int cout, float* G, int dout_ld,
                      int act_ld, int extra_ld) {
  R->n_plane = 0;
  R->has_umma = false;
  // next to the umma scheme the plane chunks are used up to 4 (measured); forced, up to the 8 of the array
  const int nc = cin / 32, max_nc = (kinds & CONV_UMMA) ? 4 : 8;
  if ((kinds & CONV_PLANE) && mode == 0 && cout == 32 && cin % 32 == 0 && nc >= 1 && nc <= max_nc) {
    bool ok = true;
    for (int c = 0; c < nc && ok; ++c) {
      if (int rc = wgrad_plane_prepare(&R->plane[c], act, B, D, H, W, cin, act_ld, c * 32, dout, dout_ld, cout, G))
        return rc;
      ok = R->plane[c].ok;
    }
    if (ok) {
      if (cin_extra) {
        if (int rc = wgrad_prepare(&R->umma, 3, extra, B, D, H, W, cin_extra, nullptr, 0, dout, cout,
                                   G + (size_t)27 * cin * cout, dout_ld, extra_ld, 0))
          return rc;
        R->has_umma = true;
      }
      R->n_plane = nc;
      return 0;
    }
  }
  if (!(kinds & CONV_UMMA)) return 0;
  if (int rc = wgrad_prepare(&R->umma, mode, act, B, D, H, W, cin, extra, cin_extra, dout, cout, G, dout_ld, act_ld,
                             extra_ld))
    return rc;
  R->has_umma = true;
  return 0;
}

int wgrad_run_enqueue(const WgradRun& R, cudaStream_t st) {
  for (int c = 0; c < R.n_plane; ++c)
    if (int e = wgrad_plane_enqueue(R.plane[c], st)) return e;
  return R.has_umma ? wgrad_enqueue(R.umma, st) : 0;
}

}  // namespace cm
