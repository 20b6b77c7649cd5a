// C-ABI front end: error reporting, layer geometry, and the lowering of nn.Conv2d / nn.ConvTranspose2d
// semantics to tap-list phases executed by conv_tc.cu (tcgen05) or conv_direct.cu (fp32 CUDA cores).
#include <mutex>

#include "internal.h"
#include "stats_ws.h"

namespace dlb {

static thread_local char g_err[512] = "";

int set_error(const char* msg) {
  snprintf(g_err, sizeof(g_err), "%s", msg);
  return DLB_ERR_INVALID;
}
int set_cuda_error(const char* where) {
  cudaError_t e = cudaGetLastError();
  snprintf(g_err, sizeof(g_err), "%s: %s", where, cudaGetErrorString(e));
  return DLB_ERR_CUDA;
}

namespace {
struct DeviceFacts { int num_sms = 0; bool smem_set[kNumSmemSlots] = {}; };
std::mutex g_facts_mu;
DeviceFacts g_facts[64];

int current_device(int* dev) {
  if (cudaGetDevice(dev) != cudaSuccess || *dev < 0 || *dev >= 64) return set_cuda_error("cudaGetDevice");
  return 0;
}
}  // namespace

int ensure_dyn_smem(const void* func, int bytes, int slot) {
  int dev = 0;
  if (current_device(&dev) != 0) return DLB_ERR_CUDA;
  std::lock_guard<std::mutex> lock(g_facts_mu);
  if (!g_facts[dev].smem_set[slot]) {
    if (cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes) != cudaSuccess)
      return set_cuda_error("cudaFuncSetAttribute(MaxDynamicSharedMemorySize)");
    g_facts[dev].smem_set[slot] = true;
  }
  return 0;
}

int device_num_sms(int* num_sms) {
  int dev = 0;
  if (current_device(&dev) != 0) return DLB_ERR_CUDA;
  std::lock_guard<std::mutex> lock(g_facts_mu);
  if (g_facts[dev].num_sms == 0 &&
      cudaDeviceGetAttribute(&g_facts[dev].num_sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
    return set_cuda_error("cudaDeviceGetAttribute(multiProcessorCount)");
  *num_sms = g_facts[dev].num_sms;
  return 0;
}

namespace {

int out_shape(const dlb_conv_desc* d, int* OH, int* OW) {
  if (d->stride != 1 && d->stride != 2) return set_error("conv: stride must be 1 or 2");
  if (d->transposed) {
    *OH = (d->H - 1) * d->stride - 2 * d->pad + d->R + d->output_padding;
    *OW = (d->W - 1) * d->stride - 2 * d->pad + d->S + d->output_padding;
  } else {
    *OH = (d->H + 2 * d->pad - d->R) / d->stride + 1;
    *OW = (d->W + 2 * d->pad - d->S) / d->stride + 1;
  }
  if (*OH < 1 || *OW < 1) return set_error("conv: empty output");
  return 0;
}

// Lower a layer to phases.  Element strides are given by (sn, sh, sw): strides of the full output tensor
// for (n, h, w) in elements (NHWC: OH*OW*C, OW*C, C; NCHW plane addressing: C*OH*OW, OW, 1).
int build_phases(const dlb_conv_desc* d, int OH, int OW, long long sn, long long sh, long long sw, PhaseGeom* out) {
  int np = 0;
  if (!d->transposed) {
    PhaseGeom& g = out[np++];
    g.N = d->N; g.H = d->H; g.W = d->W; g.OH = OH; g.OW = OW; g.stride = d->stride; g.ntaps = 0;
    g.w_taps = d->R * d->S; g.cout = d->Cout;
    for (int r = 0; r < d->R; ++r)
      for (int s = 0; s < d->S; ++s) {
        if (g.ntaps >= 64) return set_error("conv: more than 64 taps");
        g.tap_dh[g.ntaps] = r - d->pad; g.tap_dw[g.ntaps] = s - d->pad; g.tap_widx[g.ntaps] = r * d->S + s;
        ++g.ntaps;
      }
    g.ys_n = sn; g.ys_h = sh; g.ys_w = sw; g.y_base = 0;
    return np;
  }
  // ConvTranspose2d: ho = hi*stride - pad + r  =>  for output parity a: r == (a + pad) mod stride,
  // hi = i + (a + pad - r) / stride with ho = stride*i + a.  One phase per output parity class.
  const int st = d->stride;
  for (int a = 0; a < st; ++a)
    for (int b = 0; b < st; ++b) {
      PhaseGeom& g = out[np];
      g.N = d->N; g.H = d->H; g.W = d->W; g.stride = 1; g.ntaps = 0; g.w_taps = d->R * d->S; g.cout = d->Cout;
      g.OH = (OH - a + st - 1) / st; g.OW = (OW - b + st - 1) / st;
      for (int r = 0; r < d->R; ++r) {
        if (((a + d->pad - r) % st) != 0) continue;
        for (int s = 0; s < d->S; ++s) {
          if (((b + d->pad - s) % st) != 0) continue;
          g.tap_dh[g.ntaps] = (a + d->pad - r) / st; g.tap_dw[g.ntaps] = (b + d->pad - s) / st;
          g.tap_widx[g.ntaps] = r * d->S + s;
          ++g.ntaps;
        }
      }
      g.ys_n = sn; g.ys_h = sh * st; g.ys_w = sw * st; g.y_base = a * sh + b * sw;
      if (g.ntaps == 0 || g.OH < 1 || g.OW < 1) return set_error("convT: empty phase (unsupported geometry)");
      ++np;
    }
  return np;
}

}  // namespace
}  // namespace dlb

using namespace dlb;

extern "C" const char* dlb_last_error(void) { return g_err; }
extern "C" int dlb_version(void) { return 100; }

extern "C" int dlb_conv_out_shape(const dlb_conv_desc* d, int* OH, int* OW) { return out_shape(d, OH, OW); }

namespace {
struct ForkRes { cudaStream_t aux[3] = {nullptr, nullptr, nullptr}; cudaEvent_t ev_fork = nullptr; cudaEvent_t ev_join[3] = {nullptr, nullptr, nullptr}; };
thread_local ForkRes t_fork[64];
}  // namespace

extern "C" int dlb_release_thread_resources(void) {
  int keep = 0;
  cudaGetDevice(&keep);
  for (int dev = 0; dev < 64; ++dev) {
    ForkRes& fr = t_fork[dev];
    if (fr.aux[0] == nullptr && fr.ev_fork == nullptr) continue;
    cudaSetDevice(dev);
    for (int i = 0; i < 3; ++i) {
      if (fr.aux[i] != nullptr) cudaStreamDestroy(fr.aux[i]);
      if (fr.ev_join[i] != nullptr) cudaEventDestroy(fr.ev_join[i]);
    }
    if (fr.ev_fork != nullptr) cudaEventDestroy(fr.ev_fork);
    fr = ForkRes();
  }
  cudaSetDevice(keep);
  return 0;
}

struct StemSrc { const float* x; int C, S, pad, pad_mode; };

// Can the output-parity phases of this layer run as ONE launch with one TMEM accumulator per phase (halo-strip mode)?
// On success fills the merged tap list / accumulator bases and returns the UMMA N to use; 0 otherwise.
static int plan_merged(const dlb_conv_desc* d, const PhaseGeom* geo, int np, int split, int n_tile, int fa, TcPhase* out) {
  // Measured (profiles/r02_*): merging pays when all output channels fit ONE 64-wide tile with four accumulators side by
  // side (Cout <= 64: ResNet up1 0.55 -> 0.43 ms, UNet outermost 0.92 -> 0.73 ms); wider layers would need several channel
  // tiles of narrow, shared-memory-bound N = 64 MMAs and lose (Cout 128: 0.31 -> 0.38 ms, Cout 256: 0.18 -> 0.42 ms).
  if (np < 2 || np > 4 || d->Cout % 32 != 0 || d->Cout > 64) return 0;
  int total_taps = 0;
  for (int i = 0; i < np; ++i) {
    if (geo[i].OH != geo[0].OH || geo[i].OW != geo[0].OW || geo[i].stride != 1) return 0;
    total_taps += geo[i].ntaps;
  }
  if (total_taps > 16) return 0;
  int nt_m = n_tile ? n_tile : (d->Cout >= 64 ? 64 : 32);
  while (2 * np * nt_m > 512 && nt_m > 32) nt_m >>= 1;
  if (2 * np * nt_m > 512) return 0;
  TcPhase ph;
  memset(&ph, 0, sizeof(ph));
  static_cast<PhaseGeom&>(ph) = geo[0];
  ph.ntaps = 0;
  for (int i = 0; i < np; ++i) {
    for (int t = 0; t < geo[i].ntaps; ++t) {
      ph.tap_dh[ph.ntaps] = geo[i].tap_dh[t]; ph.tap_dw[ph.ntaps] = geo[i].tap_dw[t]; ph.tap_widx[ph.ntaps] = geo[i].tap_widx[t];
      ph.tap_acc[ph.ntaps] = i;
      ++ph.ntaps;
    }
    ph.acc_ybase[i] = geo[i].y_base;
  }
  ph.nacc = np;
  int tw, th, tn, nt;
  if (tc_plan_tiles(ph, d->nsrc, d->Cin, d->Cout, split, nt_m, &tw, &th, &tn, &nt, fa) != 2) return 0;
  *out = ph;
  return nt_m;
}

static int conv_tc_fwd_impl(const dlb_conv_desc* d, const void* const* x_hi, const void* const* x_lo,
                            const dlb_fused_src* fsrc, const void* w_hi, const void* w_lo, const float* bias, float* y,
                            int fmt, int split, int n_tile, void* stats_ws, size_t stats_ws_bytes, dlb_stream_t stream,
                            const StemSrc* stem = nullptr) {
  int OH, OW;
  if (out_shape(d, &OH, &OW) != 0) return DLB_ERR_INVALID;
  if (d->pad_mode != DLB_PAD_ZERO) return set_error("dlb_conv_tc_fwd: zero padding only (reflect border comes from dlb_norm_apply / dlb_fused_src.border)");
  if (d->nsrc < 1 || d->nsrc > 2) return set_error("dlb_conv_tc_fwd: nsrc must be 1 or 2");
  if (fmt != DLB_FMT_BF16 && fmt != DLB_FMT_FP16) return set_error("dlb_conv_tc_fwd: bad fmt");
  PhaseGeom geo[4];
  const long long C = d->Cout;
  const int np = build_phases(d, OH, OW, static_cast<long long>(OH) * OW * C, static_cast<long long>(OW) * C, C, geo);
  if (np < 0) return np;
  // fused statistics: one slice per 128-pixel CTA tile (the four epilogue warps merge their partials), phases concatenated
  StatsPtrs sp; memset(&sp, 0, sizeof(sp));
  int slice_base[4] = {0, 0, 0, 0}, S_total = 0;
  if (stats_ws != nullptr) {
    const StatsLayout L = stats_layout(d->N, OH * OW, d->Cout);
    if (stats_ws_bytes < L.total) return set_error("dlb_conv_tc_fwd: statistics workspace too small");
    sp = stats_ptrs(stats_ws, L);
    for (int i = 0; i < np; ++i) {
      int tw, th, tn, nt;
      tc_plan_tiles(geo[i], d->nsrc, d->Cin, d->Cout, split, n_tile, &tw, &th, &tn, &nt, fsrc != nullptr || stem != nullptr);
      if (tn != 1) return set_error("dlb_conv_tc_fwd: fused statistics need OH*OW >= 128 per phase (use dlb_norm_stats)");
      slice_base[i] = S_total;
      S_total += ((geo[i].OH + th - 1) / th) * ((geo[i].OW + tw - 1) / tw);      // one slice per 128-pixel CTA tile
    }
    if (S_total > L.S_cap) return set_error("dlb_conv_tc_fwd: statistics workspace slice capacity exceeded");
  }
  cudaStream_t main_stream = reinterpret_cast<cudaStream_t>(stream);
  auto fill_sources = [&](TcPhase& ph) -> int {
    ph.nsrc = d->nsrc;
    if (stem != nullptr) {
      ph.fa = 2; ph.fa_x[0] = stem->x; ph.stem_C = stem->C; ph.stem_S = stem->S; ph.stem_pad = stem->pad;
      ph.fa_border = 0; ph.fa_border_mode = stem->pad_mode; ph.fa_act[0] = DLB_ACT_NONE;
    }
    for (int s = 0; s < d->nsrc; ++s) {
      ph.cin[s] = d->Cin[s];
      if (stem != nullptr) continue;
      if (fsrc == nullptr) { ph.x_hi[s] = x_hi[s]; ph.x_lo[s] = split ? x_lo[s] : nullptr; continue; }
      ph.fa = 1;
      ph.fa_x[s] = fsrc[s].x; ph.fa_scale[s] = fsrc[s].scale; ph.fa_shift[s] = fsrc[s].shift; ph.fa_res[s] = fsrc[s].residual;
      ph.fa_out[s] = fsrc[s].out; ph.fa_act[s] = fsrc[s].act;
      ph.fa_border = fsrc[0].border; ph.fa_border_mode = fsrc[0].border_mode;
      if (fsrc[s].border != fsrc[0].border || fsrc[s].border_mode != fsrc[0].border_mode)
        return set_error("dlb_conv_tc_fwd_fused: every source needs the same border");
      if (fsrc[s].act != DLB_ACT_NONE && fsrc[s].act != DLB_ACT_RELU && fsrc[s].act != DLB_ACT_LRELU02)
        return set_error("dlb_conv_tc_fwd_fused: act must be none / relu / lrelu0.2");
    }
    ph.w_hi = w_hi; ph.w_lo = split ? w_lo : nullptr; ph.bias = bias; ph.y = y;
    ph.fmt = fmt; ph.split = split ? 1 : 0;
    return 0;
  };
  // ---- merged output-parity phases: the phases of a stride-2 ConvTranspose2d (and of a stride-2 data gradient) read the
  // same input; one launch loads (or converts) each input strip once and accumulates every phase in its own TMEM
  // accumulator, instead of one launch per phase each re-reading its shifted input through L2 ----
  {
    TcPhase ph;
    const int nt_m = plan_merged(d, geo, np, split, n_tile, fsrc != nullptr || stem != nullptr, &ph);
    if (nt_m > 0) {
      if (fill_sources(ph) != 0) return DLB_ERR_INVALID;
      ph.n_tile = nt_m;
      if (stats_ws != nullptr) {
        const int tiles = ((ph.OH + 15) / 16) * ((ph.OW + 7) / 8);          // halo-strip tiles: 16 x 8 output pixels
        if (np * tiles > sp.S_cap) return set_error("dlb_conv_tc_fwd: statistics workspace slice capacity exceeded");
        ph.st_partial = sp.partial; ph.st_cnt = sp.cnt; ph.st_S = sp.S; ph.st_S_cap = sp.S_cap;
        for (int i = 0; i < np; ++i) ph.acc_slice[i] = i * tiles;
        ph.st_slice_base = 0; ph.st_S_total = np * tiles;
      }
      return launch_conv_tc_phase(ph, main_stream);
    }
  }
  // The output-parity phases of a ConvTranspose2d (and of a stride-2 data gradient) are otherwise independent launches.  When one
  // phase cannot fill the GPU (inner UNet levels: a few CTAs streaming megabytes of weights, latency-bound), the
  // phases run side by side on helper streams forked from and joined back into the caller's stream (plain event
  // fork/join: also valid inside a stream capture).
  bool fork = false;
  if (np > 1) {
    int nt_eff = n_tile ? n_tile : (d->Cout >= 256 ? 256 : (d->Cout >= 128 ? 128 : (d->Cout > 32 ? 64 : 32)));
    const long long m_tiles = (static_cast<long long>(d->N) * geo[0].OH * geo[0].OW + 127) / 128;
    fork = m_tiles * ((d->Cout + nt_eff - 1) / nt_eff) < 74;
  }
  ForkRes unused;
  ForkRes* fr = &unused;
  if (fork) {
    int dev = 0;
    if (current_device(&dev) != 0) return DLB_ERR_CUDA;
    fr = &t_fork[dev];
  }
  cudaStream_t* aux = fr->aux;
  cudaEvent_t* ev_join = fr->ev_join;
  cudaEvent_t& ev_fork = fr->ev_fork;
  if (fork) {
    if (aux[0] == nullptr) {
      for (int i = 0; i < 3; ++i) {
        if (cudaStreamCreateWithFlags(&aux[i], cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&ev_join[i], cudaEventDisableTiming) != cudaSuccess) return set_cuda_error("phase streams");
      }
      if (cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming) != cudaSuccess) return set_cuda_error("phase streams");
    }
    if (cudaEventRecord(ev_fork, main_stream) != cudaSuccess) return set_cuda_error("cudaEventRecord(fork)");
    for (int i = 1; i < np; ++i)
      if (cudaStreamWaitEvent(aux[i - 1], ev_fork, 0) != cudaSuccess) return set_cuda_error("cudaStreamWaitEvent(fork)");
  }
  for (int i = 0; i < np; ++i) {
    if (geo[i].ntaps > 16) return set_error("dlb_conv_tc_fwd: more than 16 taps per phase");
    TcPhase ph;
    memset(&ph, 0, sizeof(ph));
    static_cast<PhaseGeom&>(ph) = geo[i];
    if (fill_sources(ph) != 0) return DLB_ERR_INVALID;
    ph.n_tile = n_tile;
    if (stats_ws != nullptr) {
      ph.st_partial = sp.partial; ph.st_cnt = sp.cnt; ph.st_S = sp.S; ph.st_S_cap = sp.S_cap;
      ph.st_slice_base = slice_base[i]; ph.st_S_total = S_total;
    }
    const int rc = launch_conv_tc_phase(ph, (fork && i > 0) ? aux[i - 1] : main_stream);
    if (rc != 0) return rc;
  }
  if (fork) {
    for (int i = 1; i < np; ++i) {
      if (cudaEventRecord(ev_join[i - 1], aux[i - 1]) != cudaSuccess) return set_cuda_error("cudaEventRecord(join)");
      if (cudaStreamWaitEvent(main_stream, ev_join[i - 1], 0) != cudaSuccess) return set_cuda_error("cudaStreamWaitEvent(join)");
    }
  }
  return 0;
}

extern "C" int dlb_conv_tc_launches(const dlb_conv_desc* d, int split, int n_tile, int fused) {
  int OH, OW;
  if (out_shape(d, &OH, &OW) != 0) return DLB_ERR_INVALID;
  PhaseGeom geo[4];
  const long long C = d->Cout;
  const int np = build_phases(d, OH, OW, static_cast<long long>(OH) * OW * C, static_cast<long long>(OW) * C, C, geo);
  if (np < 0) return np;
  TcPhase ph;
  return plan_merged(d, geo, np, split, n_tile, fused, &ph) > 0 ? 1 : np;
}

extern "C" int dlb_conv_tc_fused_mode(const dlb_conv_desc* d, int split, int n_tile) {
  int OH, OW;
  if (out_shape(d, &OH, &OW) != 0) return DLB_ERR_INVALID;
  if (d->nsrc < 1 || d->nsrc > 2) return set_error("dlb_conv_tc_fused_mode: nsrc must be 1 or 2");
  PhaseGeom geo[4];
  const long long C = d->Cout;
  const int np = build_phases(d, OH, OW, static_cast<long long>(OH) * OW * C, static_cast<long long>(OW) * C, C, geo);
  if (np < 0) return np;
  bool light = false, staged = d->nsrc == 1;
  int n_vs = 0;
  for (int i = 0; i < np; ++i) {
    if (geo[i].ntaps > 16) return 0;
    int tw, th, tn, nt;
    const int m = tc_plan_tiles(geo[i], d->nsrc, d->Cin, d->Cout, split, n_tile, &tw, &th, &tn, &nt, 1);
    if (m == 0) return 0;
    // tensor-pipe cycles one 64-channel chunk of this phase keeps the MMA busy: taps x 4 K-steps x (3 | 1) MMAs x N/2 cycles.
    // The converter warps need ~4-6 us per strip when they load from HBM (measured: register-staged global loads); below
    // ~8k cycles of MMA work per strip they, not the tensor pipe, set the pace — unless the source is staged by TMA.
    // (N of the widest tile the layer could use, not the planned one: the choice must not depend on the batch size, which
    // only changes how many CTAs share the work — results for a tile are then identical at every batch size.)
    const int n_wide = d->Cout >= 256 ? 256 : (d->Cout >= 128 ? 128 : (d->Cout > 32 ? 64 : 32));
    if (m == 1) { ++n_vs; light = true; }                     // resident-weight vertical strips: few taps, narrow N
    if (m == 2 && geo[i].ntaps * 4 * (split ? 3 : 1) * (n_wide / 2) < 8192) light = true;
    if (m == 2 && !hs_staging_fits(geo[i], split, nt)) staged = false;
  }
  if (np == 1 && n_vs == 1) return 1;
  if (!light) return 2;
  return staged ? 4 : 3;
}

extern "C" int dlb_conv_tc_fwd(const dlb_conv_desc* d, const void* const* x_hi, const void* const* x_lo,
                               const void* w_hi, const void* w_lo, const float* bias, float* y, int fmt, int split,
                               int n_tile, void* stats_ws, size_t stats_ws_bytes, dlb_stream_t stream) {
  return conv_tc_fwd_impl(d, x_hi, x_lo, nullptr, w_hi, w_lo, bias, y, fmt, split, n_tile, stats_ws, stats_ws_bytes, stream);
}

extern "C" int dlb_conv_tc_fwd_fused(const dlb_conv_desc* d, const dlb_fused_src* src, const void* w_hi, const void* w_lo,
                                     const float* bias, float* y, int fmt, int split, int n_tile, void* stats_ws,
                                     size_t stats_ws_bytes, dlb_stream_t stream) {
  if (src == nullptr) return set_error("dlb_conv_tc_fwd_fused: src is null");
  return conv_tc_fwd_impl(d, nullptr, nullptr, src, w_hi, w_lo, bias, y, fmt, split, n_tile, stats_ws, stats_ws_bytes, stream);
}

extern "C" int dlb_conv_tc_fwd_stem(const float* x_nchw, int N, int C, int H, int W, int pad, int S, int pad_mode, int Cout,
                                    const void* w_hi, const void* w_lo, const float* bias, float* y, int fmt, int split,
                                    int n_tile, void* stats_ws, size_t stats_ws_bytes, dlb_stream_t stream) {
  if (x_nchw == nullptr) return set_error("dlb_conv_tc_fwd_stem: x is null");
  if (S != 2 * pad + 1) return set_error("dlb_conv_tc_fwd_stem: S must be 2 * pad + 1");
  dlb_conv_desc d;
  memset(&d, 0, sizeof(d));
  d.N = N; d.H = H + 2 * pad; d.W = W; d.nsrc = 1; d.Cin[0] = 64; d.Cout = Cout; d.R = S; d.S = 1; d.stride = 1; d.pad = 0;
  d.pad_mode = DLB_PAD_ZERO;
  const StemSrc st{x_nchw, C, S, pad, pad_mode};
  return conv_tc_fwd_impl(&d, nullptr, nullptr, nullptr, w_hi, w_lo, bias, y, fmt, split, n_tile, stats_ws, stats_ws_bytes,
                          stream, &st);
}

extern "C" int dlb_conv_direct_fwd(const dlb_conv_desc* d, const float* x, int in_nchw, const float* in_scale,
                                   const float* in_shift, int in_act, const float* w_packed, const float* bias,
                                   float* y, int out_act, int out_nchw, dlb_stream_t stream) {
  if (x == nullptr) return set_error("dlb_conv_direct_fwd: x is null");
  int OH, OW;
  if (out_shape(d, &OH, &OW) != 0) return DLB_ERR_INVALID;
  if (d->nsrc != 1) return set_error("dlb_conv_direct_fwd: single source only");
  if (d->pad_mode == DLB_PAD_REFLECT && (d->transposed || d->pad >= d->H || d->pad >= d->W))
    return set_error("dlb_conv_direct_fwd: reflect padding needs a plain conv with pad < H, W");
  PhaseGeom geo[4];
  const long long C = d->Cout;
  long long sn, sh, sw, sc;
  if (out_nchw) { sn = C * OH * OW; sh = OW; sw = 1; sc = static_cast<long long>(OH) * OW; }
  else { sn = static_cast<long long>(OH) * OW * C; sh = static_cast<long long>(OW) * C; sw = C; sc = 1; }
  const int np = build_phases(d, OH, OW, sn, sh, sw, geo);
  if (np < 0) return np;
  for (int i = 0; i < np; ++i) {
    DirectPhase ph;
    memset(&ph, 0, sizeof(ph));
    static_cast<PhaseGeom&>(ph) = geo[i];
    ph.cin = d->Cin[0]; ph.x = x; ph.in_nchw = in_nchw; ph.in_scale = in_scale; ph.in_shift = in_shift;
    ph.in_act = in_act; ph.pad_mode = d->pad_mode; ph.w = w_packed; ph.bias = bias; ph.y = y; ph.out_act = out_act;
    ph.out_nchw = out_nchw; ph.ys_c = sc;
    const int rc = launch_conv_direct_phase(ph, reinterpret_cast<cudaStream_t>(stream));
    if (rc != 0) return rc;
  }
  return 0;
}
