// C ABI (include/l2s_vocoder.h) of the B200-native multi_input_vocoder generator
// forward: layer table, weight repacking, workspace carving and the launch
// sequence that replaces MelCodeGenerator.forward (models_multi_input.py:60-97) /
// Generator.forward (speech-resynthesis/models.py:98-114).
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <map>
#include <mutex>
#include <shared_mutex>
#include <string>
#include <vector>

#include "../../include/l2s_vocoder.h"
#include "../../include/l2s_debug.h"
#include "conv_common.cuh"
#include "conv_simt.cuh"
#include "conv_tc.cuh"
#include "pair_tc.cuh"
#include "frontend.cuh"
#include "res_tc.cuh"
#include "respk_tc.cuh"

using namespace l2s;

namespace {

// ------------------------------------------------------------------ knobs
struct Knobs {
  long long force_simt = 0;        // bf16 mode: run the CUDA-core kernel on the bf16 operands
  long long stop_after_stage = -1; // >= 0: stop after that MRF stage (taps stay valid)
  long long stop_after_pre = 0;    // stop after conv_pre
  long long per_tap = 0;
  long long sa_min = 0;
  long long dual = 1;
  long long span_ptr = 0;          // device array [launch][2]: min CTA start / max CTA end of every tcgen05 launch
  long long trace_launch = -1;     // index of the fused-step launch of a forward that gets trace_ptr
  long long cluster = 1;           // fused steps with C >= 128 run as CTA pairs (cluster of 2).  With cg2 (default) the pair issues
                                   // cta_group::2 MMAs: each CTA holds half of every weight stage (stage 0 -9 %, stage 1 -4 %).
                                   // Plain weight multicast (cg2 = 0) measured neutral.
  long long alias_at = 1;          // fused steps with C >= 128: A-slab ring shares the T-slab shared memory
  long long epi_tma = 0;           // dual fused steps (C <= 64, residual + raw [+ act]): TMA-streamed phase 2 (1: where it fits
                                   // without aliasing, 2: also aliased).  Bit-exact, measured neutral: TMA-store completion
                                   // latency replaces the LSU cost, so it is off by default.
  long long use_graph = 1;         // replay the conv chain (conv_pre .. last MRF stage) as a CUDA graph per (B, T, workspace)
  long long epoch = 0;             // bumped by every l2s_debug_set: cached graphs of older epochs are not reused
  long long pair_smem = 220 * 1024; // shared-memory budget of the single-CTA fused plans
  long long fuse_pairs = 1;        // bf16 mode: one kernel per ResBlock (c1, c2) step
  long long fuse_branch = 1;       // bf16 mode, C <= 64: one kernel per ResBlock (all its steps), residual stream kept in TMEM
  long long res_mode = 0;          // whole-ResBlock plans: 0 auto, 1 two CTAs per SM, 2 one CTA per SM
  long long res_msub = 8;          // whole-ResBlock plans: largest tile, in 128-row accumulators
  long long plan_report = 0;       // l2s_debug_conv: write the chosen plan + occupancy into the err buffer
  long long trace_ptr = 0;         // device pointer for the kernel trace of l2s_debug_conv (0: off)
  long long max_msub = 8;
  long long max_nt = 256;
  long long tc_cg2 = 1;            // conv_pre / upsampling convs (one CTA per SM, bf16) run as CTA pairs with cta_group::2 MMAs
  long long epi_pf = 2;            // fused-step kernels: bit 1 = L2 prefetch of the residual tile (removed: slower), bit 2 = L1 prefetch of the next
                                   // chunk's residual / branch-sum lines in the 80-register kernels (-0.4 % of the forward)
  long long slab_cap = 40960;
  long long max_ctas = 0;
  long long embed_tap = 0;
  long long layer_events = 0;      // record a cudaEvent pair around every launch of the next forwards
  long long par_share = 0;         // experiment: with branch_par, two-CTAs-per-SM step kernels launch ONE CTA per SM each, so CTAs of two
                                   // different branches (k = 3 epilogue-bound, k = 11 MMA-bound) share an SM
  long long chain = 0;             // C >= 128 stages: steps 1.. of a ResBlock are launched programmatically and consume the previous step item by
                                   // item (per-item completion counters) instead of waiting for the whole grid.  Bit-identical; measured with
                                   // tools/knob_ab.py (BURST=1): 2451 -> 2418 us per step with serial branches, but 2399 -> 2415 us next to the
                                   // parallel branch streams (branch_par, the default), which already fill the boundaries: off.  2: residual at L2.
  long long narrow_par = 0;        // C <= 64 stages run as three tap-by-tap whole-ResBlock kernels: branches 2 and 1 concurrently on two streams,
                                   // branch 0 last adding both (bit-identical; measured neutral: 2514.2 vs 2514.0 us per step in the power-capped
                                   // steady state, tools/knob_ab.py -- each kernel fills every SM, the second one only gets the first one's tail)
  long long post_rows = 1;         // head: the row-per-thread kernel (C = 16 / 32), 0: the staged-tile kernel
  long long front_fuse = 1;        // the speaker projection runs inside the conditioning kernel (0: its own launch in front of it)
  long long branch_par = 1;        // C >= 128 stages: the kernel-size branches of a stage run on parallel streams (graph branches); only the
                                   // last step of a branch waits for the previous branch (running sum).  Fills the wave-quantisation tails.
};
Knobs g_knobs;
std::shared_mutex g_knob_mu;   // forwards hold it shared, l2s_debug_set exclusively: a knob never changes under a running forward

inline uint16_t f2bf(float f) {  // round to nearest even
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}

inline float f2tf32(float f) {  // round to nearest (ties away), 10-bit mantissa, like cvt.rna.tf32.f32
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7f800000u) == 0x7f800000u) return f;
  u = (u + 0x1000u) & 0xffffe000u;
  memcpy(&f, &u, 4);
  return f;
}

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct ConvLayer {
  std::string name;
  bool transposed = false;
  int cin = 0, cout = 0, k = 0, dil = 1, up = 1, pad = 0;
  int cin_pad = 0, ntaps = 0, ntot = 0;
  int tap_off[kMaxTaps] = {0};
  long long out_shift = 0;
  void* w_dev = nullptr;       // [ntaps][ntot][cin_pad] fp32 or bf16
  float* bias_dev = nullptr;   // [ntot]
  CUtensorMap tmW;
  bool has_tmW = false;
  int tm_nt = 0, tm_tb = 0;
  // time-packed whole-ResBlock kernel (respk_tc.cuh): block-Toeplitz copy [pk_groups][128][64] bf16
  void* wpk_dev = nullptr;
  int pk_groups = 0;
  CUtensorMap tmWpk;
  int tmpk_rows = 0, tmpk_tb = 0;
};

}  // namespace

struct l2s_vocoder {
  l2s_config cfg;
  std::map<std::string, std::vector<float>> weights;
  std::map<std::string, long long> expected;   // name -> numel
  std::vector<ConvLayer> convs;                // conv_pre, then per stage: ups, 3 x 3 x (c1, c2)
  int conv_pre = -1;
  std::vector<int> ups;                        // index into convs
  std::vector<std::vector<std::vector<int>>> rb_c1, rb_c2;  // [stage][branch][dil]
  std::vector<int> stage_ch;
  float* d_zero_bias = nullptr;                // 256 zeros: output epilogue of the whole-ResBlock kernel
  std::vector<std::vector<float*>> pk_bias;    // [stage][branch]: [kPkBiasRows][128] per-column constants of the time-packed kernel
  std::vector<float*> pk_bias_stage;           // [stage]: the same for all branches back to back, [n_rk][kPkBiasRows][128]
  std::vector<char> pk_ok;                     // [stage]: config-only: the time-packed kernel can run this stage (set by l2s_create)
  std::vector<std::vector<std::vector<float>>> pk_bias_host;   // [stage][branch]: [kPkBiasRows][64] per-channel copy handed to the kernel by value
  bool finalized = false;
  int device = -1, num_sms = 0;
  // device-side small weights
  float* d_unit_tab = nullptr;   // [4][num_embeddings][E]: the unit table folded through the ConvTranspose1d taps
  float *d_dict = nullptr, *d_spk_w = nullptr, *d_spk_b = nullptr, *d_wt = nullptr, *d_wt_b = nullptr, *d_fc_t = nullptr,
        *d_fc_b = nullptr, *d_post_w = nullptr;
  float post_bias = 0.f;
  std::vector<float> post_w_host;   // conv_post weights [7][C], handed to the kernel by value
  int* err_host = nullptr;   // mapped pinned
  int* err_dev = nullptr;
  std::vector<void*> dev_allocs;
  std::string err;
  std::mutex mu;
  // last-forward bookkeeping for taps
  struct Tap { const void* ptr; long long numel; bool act; };
  std::map<std::string, Tap> taps;
  // optional per-launch timing (l2s_debug_set("layer_events", 1))
  struct Timed { std::string name; cudaEvent_t a, b; double flops; };
  std::vector<Timed> timed;
  size_t timed_used = 0;
  long long pair_launches = 0;     // fused-step launches issued by the current forward
  long long res_launches = 0;      // whole-ResBlock launches issued by the current forward
  long long tc_launches = 0;       // all tcgen05 launches of the current forward (span_ptr slots)
  // CUDA-graph replay of the conv chain
  struct ChainGraph { int batch, frames; void* workspace; long long epoch; int seen; cudaGraphExec_t exec; };
  std::vector<ChainGraph> graphs;
  cudaStream_t capture_stream = nullptr;
  cudaStream_t br_stream[L2S_MAX_RK] = {nullptr};   // parallel branches of a stage (index 0 unused: branch 0 stays on the caller's stream)
  cudaEvent_t ev_fork = nullptr, ev_acc[L2S_MAX_RK] = {nullptr}, ev_join[L2S_MAX_RK] = {nullptr};
};

namespace {

int fail(l2s_vocoder* v, int code, const std::string& msg) {
  if (v) v->err = msg;
  return code;
}

bool is_bf16(const l2s_vocoder* v) { return v->cfg.precision == L2S_PREC_BF16; }
bool is_tf32(const l2s_vocoder* v) { return v->cfg.precision == L2S_PREC_TF32; }
size_t act_size(const l2s_vocoder* v) { return is_bf16(v) ? 2 : 4; }

int hop_of(const l2s_config& c) {
  int h = 1;
  for (int i = 0; i < c.n_ups; ++i) h *= c.up_rates[i];
  return h;
}

ConvLayer make_conv(const std::string& name, int cin, int cout, int k, int dil) {
  ConvLayer L;
  L.name = name;
  L.cin = cin; L.cout = cout; L.k = k; L.dil = dil;
  L.cin_pad = cin <= 64 ? (int)align_up(cin, 16) : (int)align_up(cin, 64);
  L.ntaps = k;
  L.ntot = cout;
  for (int j = 0; j < k; ++j) L.tap_off[j] = (j - (k - 1) / 2) * dil;
  L.out_shift = 0;
  return L;
}

ConvLayer make_convT(const std::string& name, int cin, int cout, int k, int u, int p) {
  ConvLayer L;
  L.name = name;
  L.transposed = true;
  L.cin = cin; L.cout = cout; L.k = k; L.up = u; L.pad = p;
  L.cin_pad = cin <= 64 ? (int)align_up(cin, 16) : (int)align_up(cin, 64);
  L.ntaps = (k + u - 1) / u;
  L.ntot = u * cout;
  for (int m = 0; m < L.ntaps; ++m) L.tap_off[m] = -m;
  L.out_shift = -(long long)p * cout;
  return L;
}

int build_layers(l2s_vocoder* v) {
  const l2s_config& c = v->cfg;
  if (c.n_ups < 1 || c.n_ups > L2S_MAX_UPS || c.n_rk < 1 || c.n_rk > L2S_MAX_RK || c.n_dil < 1 || c.n_dil > L2S_MAX_DIL)
    return fail(v, L2S_ERR_INVALID, "bad layer counts");
  if (c.precision != L2S_PREC_FP32 && c.precision != L2S_PREC_BF16 && c.precision != L2S_PREC_TF32)
    return fail(v, L2S_ERR_INVALID, "bad precision");
  if (c.embedding_dim != kCondE) return fail(v, L2S_ERR_UNSUPPORTED, "embedding_dim must be 128");
  if (c.num_embeddings < 1) return fail(v, L2S_ERR_INVALID, "num_embeddings");
  const int E = c.embedding_dim;
  int in_dim;
  if (c.variant == L2S_VARIANT_MULTI_INPUT) {
    if (c.num_mels < 1) return fail(v, L2S_ERR_INVALID, "num_mels");
    if (c.multispkr && c.spk_dim <= 0) return fail(v, L2S_ERR_UNSUPPORTED, "multi-input needs embedder_dim (speaker Linear)");
    in_dim = c.num_mels + E + (c.multispkr ? E : 0);
  } else if (c.variant == L2S_VARIANT_UNIT_ONLY) {
    if (c.multispkr && c.num_speakers < 1) return fail(v, L2S_ERR_INVALID, "num_speakers");
    in_dim = E + (c.multispkr ? E : 0);
  } else {
    return fail(v, L2S_ERR_INVALID, "bad variant");
  }
  if (c.model_in_dim != in_dim) {
    char b[128];
    snprintf(b, sizeof b, "model_in_dim %d does not match the conditioning channels %d", c.model_in_dim, in_dim);
    return fail(v, L2S_ERR_SHAPE, b);
  }
  int ch = c.up_init_ch;
  if (ch % 16 != 0) return fail(v, L2S_ERR_UNSUPPORTED, "upsample_initial_channel must be a multiple of 16");
  v->convs.clear();
  v->pk_ok.clear();
  v->convs.push_back(make_conv("conv_pre", in_dim, ch, 7, 1));
  v->conv_pre = 0;
  v->expected["conv_pre.weight"] = (long long)ch * in_dim * 7;
  v->expected["conv_pre.bias"] = ch;
  for (int i = 0; i < c.n_ups; ++i) {
    const int u = c.up_rates[i], k = c.up_ksizes[i];
    if (u < 1 || k < u || (k - u) % 2 != 0) return fail(v, L2S_ERR_UNSUPPORTED, "upsample kernel/rate: need k >= u and k-u even");
    if ((k + u - 1) / u > kMaxTaps) return fail(v, L2S_ERR_UNSUPPORTED, "too many polyphase taps");
    if (ch % 2 != 0 || (ch / 2) % 16 != 0) return fail(v, L2S_ERR_UNSUPPORTED, "stage channels must stay multiples of 16");
    char nm[64];
    snprintf(nm, sizeof nm, "ups.%d", i);
    v->convs.push_back(make_convT(nm, ch, ch / 2, k, u, (k - u) / 2));
    v->ups.push_back((int)v->convs.size() - 1);
    v->expected[std::string(nm) + ".weight"] = (long long)ch * (ch / 2) * k;
    v->expected[std::string(nm) + ".bias"] = ch / 2;
    ch /= 2;
    v->stage_ch.push_back(ch);
    v->pk_ok.push_back(c.precision == L2S_PREC_BF16 && c.n_dil <= kPkMaxDil && (ch == 16 || ch == 32 || ch == 64) ? 1 : 0);
    std::vector<std::vector<int>> s1, s2;
    for (int j = 0; j < c.n_rk; ++j) {
      const int rk = c.rk_sizes[j];
      if (rk < 1 || rk > kMaxTaps || rk % 2 == 0) return fail(v, L2S_ERR_UNSUPPORTED, "resblock kernel sizes must be odd and <= 16");
      std::vector<int> b1, b2;
      for (int m = 0; m < c.n_dil; ++m) {
        const int n = i * c.n_rk + j;
        snprintf(nm, sizeof nm, "resblocks.%d.convs1.%d", n, m);
        v->convs.push_back(make_conv(nm, ch, ch, rk, c.rk_dils[j][m]));
        b1.push_back((int)v->convs.size() - 1);
        v->expected[std::string(nm) + ".weight"] = (long long)ch * ch * rk;
        v->expected[std::string(nm) + ".bias"] = ch;
        snprintf(nm, sizeof nm, "resblocks.%d.convs2.%d", n, m);
        v->convs.push_back(make_conv(nm, ch, ch, rk, 1));
        b2.push_back((int)v->convs.size() - 1);
        v->expected[std::string(nm) + ".weight"] = (long long)ch * ch * rk;
        v->expected[std::string(nm) + ".bias"] = ch;
      }
      s1.push_back(b1);
      s2.push_back(b2);
    }
    v->rb_c1.push_back(s1);
    v->rb_c2.push_back(s2);
  }
  if (ch > 64) return fail(v, L2S_ERR_UNSUPPORTED, "final channel count must be <= 64");
  // Every conv reads its input rows with pitch cin_pad, but the epilogues write activations with pitch cout and the
  // workspace holds len * ch elements per stage.  Only the front end writes conv_pre's input with the padded pitch, so
  // any other layer whose input channels get padded (C > 64 and not a multiple of 64) would read misaligned rows.
  for (const ConvLayer& L : v->convs) {
    if (&L == &v->convs[v->conv_pre] || L.cin_pad == L.cin) continue;
    char b[160];
    snprintf(b, sizeof b, "%s has %d input channels: channel counts above 64 must be multiples of 64", L.name.c_str(), L.cin);
    return fail(v, L2S_ERR_UNSUPPORTED, b);
  }
  v->expected["conv_post.weight"] = (long long)ch * 7;
  v->expected["conv_post.bias"] = 1;
  v->expected["dict.weight"] = (long long)c.num_embeddings * E;
  if (c.variant == L2S_VARIANT_MULTI_INPUT) {
    v->expected["layer.0.weight"] = (long long)E * E * 4;
    v->expected["layer.0.bias"] = E;
    v->expected["fc.weight"] = (long long)E * E;
    v->expected["fc.bias"] = E;
    if (c.multispkr) {
      v->expected["spkr.weight"] = (long long)E * c.spk_dim;
      v->expected["spkr.bias"] = E;
    }
  } else if (c.multispkr) {
    v->expected["spkr.weight"] = (long long)c.num_speakers * E;
  }
  return L2S_OK;
}

template <typename T>
T* dev_upload(l2s_vocoder* v, const T* host, size_t n, cudaError_t* e) {
  void* d = nullptr;
  *e = cudaMalloc(&d, n * sizeof(T) > 0 ? n * sizeof(T) : 16);
  if (*e != cudaSuccess) return nullptr;
  v->dev_allocs.push_back(d);
  *e = cudaMemcpy(d, host, n * sizeof(T), cudaMemcpyHostToDevice);
  return reinterpret_cast<T*>(d);
}

// [ntaps][ntot][cin_pad] from the PyTorch layouts.
void pack_conv(const ConvLayer& L, const std::vector<float>& w, const std::vector<float>& b, std::vector<float>* pw,
               std::vector<float>* pb) {
  pw->assign((size_t)L.ntaps * L.ntot * L.cin_pad, 0.f);
  pb->assign((size_t)L.ntot, 0.f);
  if (!L.transposed) {
    // Conv1d weight (Cout, Cin, k)
    for (int co = 0; co < L.cout; ++co)
      for (int ci = 0; ci < L.cin; ++ci)
        for (int j = 0; j < L.k; ++j)
          (*pw)[((size_t)j * L.ntot + co) * L.cin_pad + ci] = w[((size_t)co * L.cin + ci) * L.k + j];
    for (int co = 0; co < L.cout; ++co) (*pb)[co] = b[co];
  } else {
    // ConvTranspose1d weight (Cin, Cout, k); column r*Cout+co of tap m holds W[ci][co][r + m*u]
    for (int m = 0; m < L.ntaps; ++m)
      for (int r = 0; r < L.up; ++r) {
        const int j = r + m * L.up;
        if (j >= L.k) continue;
        for (int co = 0; co < L.cout; ++co)
          for (int ci = 0; ci < L.cin; ++ci)
            (*pw)[((size_t)m * L.ntot + r * L.cout + co) * L.cin_pad + ci] = w[((size_t)ci * L.cout + co) * L.k + j];
      }
    for (int r = 0; r < L.up; ++r)
      for (int co = 0; co < L.cout; ++co) (*pb)[(size_t)r * L.cout + co] = b[co];
  }
}

TcTune current_tune(const l2s_vocoder* v) {
  TcTune t;
  t.max_msub = (int)g_knobs.max_msub;
  t.max_nt = (int)g_knobs.max_nt;
  t.cg2 = (int)g_knobs.tc_cg2;
  t.slab_cap = (int)g_knobs.slab_cap;
  t.per_tap = (int)g_knobs.per_tap;
  t.sa_min = (int)g_knobs.sa_min;
  t.dual = (int)g_knobs.dual;
  t.max_ctas = g_knobs.max_ctas > 0 ? (int)g_knobs.max_ctas : (v ? v->num_sms : 148);
  return t;
}

void timed_begin(l2s_vocoder* v, cudaStream_t st, const std::string& name, double flops) {
  if (!g_knobs.layer_events) return;
  if (v->timed_used == v->timed.size()) {
    l2s_vocoder::Timed t;
    cudaEventCreate(&t.a);
    cudaEventCreate(&t.b);
    v->timed.push_back(t);
  }
  l2s_vocoder::Timed& t = v->timed[v->timed_used];
  t.name = name;
  t.flops = flops;
  cudaEventRecord(t.a, st);
}
void timed_end(l2s_vocoder* v, cudaStream_t st) {
  if (!g_knobs.layer_events) return;
  cudaEventRecord(v->timed[v->timed_used].b, st);
  ++v->timed_used;
}

// One conv launch in the handle's precision mode.
int run_conv(l2s_vocoder* v, ConvLayer& L, cudaStream_t st, int batch, int lin, const void* in, float* out_raw,
             void* out_act, const float* res, const float* acc_in, float div, float slope) {
  ConvParams p{};
  p.in = in;
  p.w = L.w_dev;
  p.bias = L.bias_dev;
  p.out_raw = out_raw;
  p.out_act = out_act;
  p.res = res;
  p.acc_in = acc_in;
  p.batch = batch;
  p.lin = lin;
  p.cin_pad = L.cin_pad;
  p.ntaps = L.ntaps;
  p.ntot = L.ntot;
  // polyphase ConvTranspose1d: output n = q u + r - p; the last output (n = lin u - 1, r = 0) sits in row q = lin + ceil(p / u) - 1
  p.mrows = L.transposed ? lin + (L.pad + L.up - 1) / L.up : lin;
  for (int j = 0; j < L.ntaps; ++j) p.tap_off[j] = L.tap_off[j];
  p.out_shift = L.out_shift;
  p.out_valid = (long long)lin * L.up * L.cout;
  p.div = div;
  p.slope = slope;
  cudaError_t e;
  timed_begin(v, st, L.name, 2.0 * L.cin * L.cout * L.k * (double)batch * lin);
  p.act_f32 = is_tf32(v) ? 1 : 0;
  if (v->cfg.precision == L2S_PREC_FP32 || (is_tf32(v) && g_knobs.force_simt)) {
    e = launch_conv_simt<float>(p, st);
  } else if (g_knobs.force_simt) {
    e = launch_conv_simt<__nv_bfloat16>(p, st);
  } else {
    TcTune tune = current_tune(v);
    TcGeom g;
    if (!tc_plan(p, batch, tune, &g)) return fail(v, L2S_ERR_UNSUPPORTED, "no tcgen05 plan for " + L.name);
    const int w_rows = g.cg2 ? g.nt / 2 : g.nt;   // CTA pairs: each CTA loads half of a stage's output-channel rows
    if (!L.has_tmW || L.tm_nt != w_rows || L.tm_tb != g.tb) {
      if (!make_tmap_3d(&L.tmW, L.w_dev, g.esz, (uint64_t)L.cin_pad, (uint64_t)L.ntot, (uint64_t)L.ntaps,
                        (uint32_t)(g.rb / g.esz), (uint32_t)w_rows, (uint32_t)g.tb))
        return fail(v, L2S_ERR_CUDA, "cuTensorMapEncodeTiled failed for the weights of " + L.name);
      L.has_tmW = true;
      L.tm_nt = w_rows;
      L.tm_tb = g.tb;
    }
    CUtensorMap tmA;
    if (!make_tmap_3d(&tmA, in, g.esz, (uint64_t)L.cin_pad, (uint64_t)lin, (uint64_t)batch, (uint32_t)(g.rb / g.esz),
                      (uint32_t)g.box_rows, 1u))
      return fail(v, L2S_ERR_CUDA, "cuTensorMapEncodeTiled failed for the input of " + L.name);
    unsigned long long* span = g_knobs.span_ptr ? reinterpret_cast<unsigned long long*>(g_knobs.span_ptr) + 2 * v->tc_launches : nullptr;
    ++v->tc_launches;
    e = launch_conv_tc(p, g, tmA, L.tmW, tune.max_ctas, st, nullptr, span);
  }
  timed_end(v, st);
  if (e != cudaSuccess) return fail(v, L2S_ERR_CUDA, std::string("launch ") + L.name + ": " + cudaGetErrorString(e));
  return L2S_OK;
}

bool ensure_w_map(ConvLayer& L, int rb, int nt, int tb) {
  if (L.has_tmW && L.tm_nt == nt && L.tm_tb == tb) return true;
  if (!make_tmap_bf16_3d(&L.tmW, L.w_dev, (uint64_t)L.cin_pad, (uint64_t)L.ntot, (uint64_t)L.ntaps, (uint32_t)(rb / 2),
                         (uint32_t)nt, (uint32_t)tb))
    return false;
  L.has_tmW = true;
  L.tm_nt = nt;
  L.tm_tb = tb;
  return true;
}

bool pairs_fused(const l2s_vocoder* v) { return is_bf16(v) && !g_knobs.force_simt && g_knobs.fuse_pairs; }

// One fused ResBlock step  y = x + c2(lrelu(c1(xa)))  (bf16 tensor-core mode).  Returns
// L2S_ERR_UNSUPPORTED when no fused plan exists (the caller then runs the two convs).
int run_pair(l2s_vocoder* v, ConvLayer& c1, ConvLayer& c2, cudaStream_t st, int batch, int lin, const void* in_act,
             const float* res, float* out_raw, void* out_act, const float* acc_in, float div, float slope,
             const int* wait_flags = nullptr, int* done_flags = nullptr) {
  if (c1.cin != c1.cout || c2.cin != c2.cout || c1.cin != c2.cin || c1.cin_pad != c1.cin || c1.k != c2.k || c2.dil != 1)
    return L2S_ERR_UNSUPPORTED;
  PairGeom g;
  const int emode = (res ? kEpiRes : 0) | ((acc_in || div != 1.0f) ? kEpiAcc : 0) | (out_raw ? kEpiRaw : 0) | (out_act ? kEpiAct : 0);
  const bool want_tma = g_knobs.epi_tma != 0 && (emode == 5 || emode == 13);
  if (!pair_plan(c1.cin, c1.k, c1.dil, lin, batch, (int)g_knobs.pair_smem, g_knobs.dual != 0, g_knobs.cluster != 0, g_knobs.alias_at != 0,
                 want_tma, g_knobs.epi_tma == 2, &g))
    return L2S_ERR_UNSUPPORTED;
  // with CTA-pair multicast each CTA fetches half of the output-channel rows of a weight stage
  if (!ensure_w_map(c1, g.rb, g.c / g.cluster, g.tb) || !ensure_w_map(c2, g.rb, g.c / g.cluster, g.tb))
    return fail(v, L2S_ERR_CUDA, "cuTensorMapEncodeTiled failed for the weights of " + c1.name);
  CUtensorMap tmA;
  if (!make_tmap_bf16_3d(&tmA, in_act, (uint64_t)c1.cin_pad, (uint64_t)lin, (uint64_t)batch, (uint32_t)(g.rb / 2),
                         (uint32_t)g.box_rows, 1u))
    return fail(v, L2S_ERR_CUDA, "cuTensorMapEncodeTiled failed for the input of " + c1.name);
  ConvParams p{};
  p.in = in_act;
  p.w = c2.w_dev;
  p.bias = c2.bias_dev;
  p.out_raw = out_raw;
  p.out_act = out_act;
  p.res = res;
  p.acc_in = acc_in;
  p.batch = batch;
  p.lin = lin;
  p.cin_pad = c2.cin_pad;
  p.ntaps = c2.ntaps;
  p.ntot = c2.ntot;
  p.mrows = lin;
  p.out_shift = 0;
  p.out_valid = (long long)lin * c2.cout;
  p.div = div;
  p.slope = slope;
  // chained step: the residual rows come from a grid that may still be running.  Plain (L1) loads are sound: the producer warp's
  // ld.acquire.gpu of the item's counters precedes them in causality order (TMA -> mbarrier -> MMA -> commit -> epilogue wait);
  // knob chain = 2 reads them at L2 instead (bit 4 of pf).
  p.pf = (int)g_knobs.epi_pf | ((wait_flags && g_knobs.chain == 2) ? 4 : 0);
  timed_begin(v, st, c1.name + "+c2", 4.0 * c1.cin * c1.cout * c1.k * (double)batch * lin);
  int ctas = g_knobs.max_ctas > 0 ? (int)g_knobs.max_ctas : v->num_sms;
  if (g_knobs.par_share && g_knobs.branch_par && g.dual) ctas = (ctas + 1) / 2;   // launch_pair_tc doubles it for dual plans
  PairEpiMaps em{};
  if (g.epi_tma) {
    const int tail_rows = 32 - 2 * g.h2 > 0 ? 32 - 2 * g.h2 : 32;
    const uint64_t C = (uint64_t)c2.cout, L = (uint64_t)lin, B = (uint64_t)batch;
    bool ok = make_tmap_3d(&em.res, res, 4, C, L, B, 16u, 32u, 1u) && make_tmap_3d(&em.raw, out_raw, 4, C, L, B, 16u, 32u, 1u) &&
              make_tmap_3d(&em.raw_tail, out_raw, 4, C, L, B, 16u, (uint32_t)tail_rows, 1u);
    if (out_act)
      ok = ok && make_tmap_3d(&em.act, out_act, 2, C, L, B, 16u, 32u, 1u) &&
           make_tmap_3d(&em.act_tail, out_act, 2, C, L, B, 16u, (uint32_t)tail_rows, 1u);
    else { em.act = em.raw; em.act_tail = em.raw_tail; }
    if (!ok) return fail(v, L2S_ERR_CUDA, "cuTensorMapEncodeTiled failed for the epilogue tensors of " + c1.name);
  } else {
    em.res = tmA; em.raw = tmA; em.raw_tail = tmA; em.act = tmA; em.act_tail = tmA;   // never read
  }
  long long* trace = (g_knobs.trace_ptr && g_knobs.trace_launch == v->pair_launches) ? reinterpret_cast<long long*>(g_knobs.trace_ptr) : nullptr;
  ++v->pair_launches;
  unsigned long long* span = g_knobs.span_ptr ? reinterpret_cast<unsigned long long*>(g_knobs.span_ptr) + 2 * v->tc_launches : nullptr;
  ++v->tc_launches;
  if (g.epi_tma) { wait_flags = nullptr; done_flags = nullptr; }   // TMA-store epilogue: its completion is not covered by the flags
  cudaError_t e = launch_pair_tc(p, c1.bias_dev, g, tmA, c1.tmW, c2.tmW, em, ctas, st, trace, span, wait_flags, done_flags);
  timed_end(v, st);
  if (e != cudaSuccess) return fail(v, L2S_ERR_CUDA, std::string("launch pair ") + c1.name + ": " + cudaGetErrorString(e));
  return L2S_OK;
}

bool branch_geom(const l2s_vocoder* v, int i, int j, int lin, int batch, ResGeom* g) {
  const l2s_config& c = v->cfg;
  const ConvLayer& a = v->convs[v->rb_c1[i][j][0]];
  int dil[kResMaxDil];
  if (c.n_dil > kResMaxDil || a.cin != a.cout || a.cin_pad != a.cin) return false;
  for (int m = 0; m < c.n_dil; ++m) {
    const ConvLayer& a1 = v->convs[v->rb_c1[i][j][m]];
    const ConvLayer& a2 = v->convs[v->rb_c2[i][j][m]];
    if (a1.k != a.k || a2.k != a.k || a2.dil != 1) return false;
    dil[m] = a1.dil;
  }
  return res_plan(a.cin, a.k, c.n_dil, dil, lin, batch, (int)g_knobs.res_mode, (int)g_knobs.res_msub, g);
}

// Time-packed plan of branches [j0, j0 + n_br) of stage i, if there is one (respk_tc.cuh).
bool branch_pk_geom(const l2s_vocoder* v, int i, int j0, int n_br, int lin, int batch, PkGeom* g) {
  const l2s_config& c = v->cfg;
  int dil[kPkMaxDil], ks[kPkMaxBr];
  if (c.n_dil > kPkMaxDil || n_br < 1 || n_br > kPkMaxBr || !v->pk_ok[i]) return false;
  const int ch = v->stage_ch[i];
  for (int j = j0; j < j0 + n_br; ++j) {
    const ConvLayer& a = v->convs[v->rb_c1[i][j][0]];
    if (a.cin != a.cout || a.cin_pad != a.cin || a.cin != ch) return false;
    ks[j - j0] = a.k;
    for (int m = 0; m < c.n_dil; ++m) {
      const ConvLayer& a1 = v->convs[v->rb_c1[i][j][m]];
      const ConvLayer& a2 = v->convs[v->rb_c2[i][j][m]];
      if (a1.k != a.k || a2.k != a.k || a2.dil != 1) return false;
      if (j == j0) dil[m] = a1.dil;
      else if (dil[m] != a1.dil) return false;              // fused branches share the phase-major layouts
    }
  }
  return pk_plan(ch, n_br, ks, c.n_dil, dil, lin, batch, g);
}

// All branches of stage i in one time-packed launch?
bool stage_pk_fused(const l2s_vocoder* v, int i, int lin, int batch, PkGeom* g) {
  return g_pk_fuse_br && v->cfg.n_rk >= 2 && v->cfg.n_rk <= kPkMaxBr && branch_pk_geom(v, i, 0, v->cfg.n_rk, lin, batch, g);
}

// Every ResBlock of stage i runs as one whole-ResBlock kernel (bf16 mode, C <= 64, a plan exists for each branch).
bool stage_branch_fused(const l2s_vocoder* v, int i, int lin, int batch) {
  if (!pairs_fused(v) || !g_knobs.fuse_branch || v->stage_ch[i] > 64) return false;
  for (int j = 0; j < v->cfg.n_rk; ++j) {
    ResGeom g;
    PkGeom pg;
    if (!branch_pk_geom(v, i, j, 1, lin, batch, &pg) && !branch_geom(v, i, j, lin, batch, &g)) return false;
  }
  return true;
}

// Branches [j0, j0 + n_br) of stage i through the time-packed kernel (n_br > 1: one launch, the branches run back to back
// on every tile and the running branch sum goes through acc_buf).  out_raw / out_act / acc_in / div describe the output
// of the LAST branch.  L2S_ERR_UNSUPPORTED: no packed plan (the caller runs the tap-by-tap kernel per branch).
int run_respk(l2s_vocoder* v, int i, int j0, int n_br, cudaStream_t st, int batch, int lin, const float* x, float* out_raw, void* out_act,
              const float* acc_in, float* acc_buf, float div, float slope) {
  const l2s_config& c = v->cfg;
  PkParams P{};
  if (!branch_pk_geom(v, i, j0, n_br, lin, batch, &P.g)) return L2S_ERR_UNSUPPORTED;
  if (!pk_mode_supported(((acc_in || div != 1.0f) ? kEpiAcc : 0) | (out_raw ? kEpiRaw : 0) | (out_act ? kEpiAct : 0))) return L2S_ERR_UNSUPPORTED;
  if (!v->finalized || !v->pk_bias[i][j0] || (n_br > 1 && (j0 != 0 || !v->pk_bias_stage[i] || !acc_buf))) return L2S_ERR_UNSUPPORTED;
  const PkGeom& g = P.g;
  PkMaps maps;
  double flops = 0.0;
  const int w_rows = g.cg2 ? 64 : 128;
  for (int br = 0; br < n_br; ++br)
    for (int m = 0; m < c.n_dil; ++m)
      for (int which = 0; which < 2; ++which) {
        ConvLayer& L = v->convs[which ? v->rb_c2[i][j0 + br][m] : v->rb_c1[i][j0 + br][m]];
        if (L.tmpk_rows != w_rows || L.tmpk_tb != g.tb) {
          if (!make_tmap_bf16_3d(&L.tmWpk, L.wpk_dev, 64u, 128u, (uint64_t)L.pk_groups, 64u, (uint32_t)w_rows, (uint32_t)g.tb))
            return fail(v, L2S_ERR_CUDA, "cuTensorMapEncodeTiled failed for the packed weights of " + L.name);
          L.tmpk_rows = w_rows;
          L.tmpk_tb = g.tb;
        }
        maps.w[br * 2 * kPkMaxDil + 2 * m + which] = L.tmWpk;
        flops += 2.0 * L.cin * L.cout * L.k * (double)batch * lin;
      }
  for (int m = 0; m < kPkMaxBr * 2 * kPkMaxDil; ++m)
    if (m / (2 * kPkMaxDil) >= n_br || m % (2 * kPkMaxDil) >= 2 * c.n_dil) maps.w[m] = maps.w[0];
  const float* cols = n_br > 1 ? v->pk_bias_stage[i] : v->pk_bias[i][j0];      // [n_br][kPkBiasRows][128]
  ConvParams& p = P.c;                        // output epilogue in packed terms: rows = blocks of P time steps, 128 columns
  p.bias = cols + (size_t)((n_br - 1) * kPkBiasRows + 2 * kPkMaxDil) * 128;
  p.out_raw = out_raw;
  p.out_act = out_act;
  p.acc_in = n_br > 1 ? acc_buf : acc_in;
  p.batch = batch;
  p.lin = lin / g.P;
  p.cin_pad = 128;
  p.ntaps = 1;
  p.ntot = 128;
  p.mrows = lin / g.P;
  p.out_shift = 0;
  p.out_valid = (long long)lin * g.c;
  p.div = div;
  p.slope = slope;
  P.x = x;
  P.bias_cols = cols;
  P.acc_buf = acc_buf;
  for (int br = 0; br < n_br; ++br) memcpy(P.bias_ch[br], v->pk_bias_host[i][j0 + br].data(), sizeof(P.bias_ch[br]));
  P.lin = lin;
  P.span = g_knobs.span_ptr ? reinterpret_cast<unsigned long long*>(g_knobs.span_ptr) + 2 * v->tc_launches : nullptr;
  ++v->tc_launches;
  P.trace = (g_knobs.trace_ptr && g_knobs.trace_launch == v->res_launches) ? reinterpret_cast<long long*>(g_knobs.trace_ptr) : nullptr;
  ++v->res_launches;
  const std::string nm = v->convs[v->rb_c1[i][j0][0]].name;
  timed_begin(v, st, nm.substr(0, nm.find(".convs1")) + (n_br > 1 ? " (packed x" + std::to_string(n_br) + ")" : " (packed)"), flops);
  const int ctas = g_knobs.max_ctas > 0 ? (int)g_knobs.max_ctas : v->num_sms;
  cudaError_t e = launch_respk_tc(P, maps, ctas, st);
  timed_end(v, st);
  if (e != cudaSuccess) return fail(v, L2S_ERR_CUDA, std::string("launch packed ResBlock ") + nm + ": " + cudaGetErrorString(e));
  return L2S_OK;
}

// One whole ResBlock: x -> x + sum of its steps, then the branch sum / mean epilogue.
int run_res(l2s_vocoder* v, int i, int j, cudaStream_t st, int batch, int lin, const float* x, float* out_raw, void* out_act,
            const float* acc_in, float div, float slope, const float* acc_in2 = nullptr) {
  const l2s_config& c = v->cfg;
  ResParams P{};
  if (!branch_geom(v, i, j, lin, batch, &P.g)) return L2S_ERR_UNSUPPORTED;
  const ResGeom& g = P.g;
  ResMaps maps;
  double flops = 0.0;
  for (int m = 0; m < c.n_dil; ++m) {
    ConvLayer& c1 = v->convs[v->rb_c1[i][j][m]];
    ConvLayer& c2 = v->convs[v->rb_c2[i][j][m]];
    const int w_rows = g.cg2 ? g.c / 2 : g.c;   // CTA pairs: each CTA loads half of the output-channel rows of a stage
    if (!ensure_w_map(c1, g.rb, w_rows, g.tb) || !ensure_w_map(c2, g.rb, w_rows, g.tb))
      return fail(v, L2S_ERR_CUDA, "cuTensorMapEncodeTiled failed for the weights of " + c1.name);
    maps.w[2 * m] = c1.tmW;
    maps.w[2 * m + 1] = c2.tmW;
    P.bias1[m] = c1.bias_dev;
    P.bias2[m] = c2.bias_dev;
    flops += 4.0 * c1.cin * c1.cout * c1.k * (double)batch * lin;
  }
  for (int m = 2 * c.n_dil; m < 2 * kResMaxDil; ++m) maps.w[m] = maps.w[0];
  ConvParams& p = P.c;
  p.bias = v->d_zero_bias;   // the kernel folds every bias into its TMEM-resident stream
  p.out_raw = out_raw;
  p.out_act = out_act;
  p.acc_in = acc_in;
  p.res = acc_in2;           // the output of a second, parallel branch (added before the running sum)
  p.batch = batch;
  p.lin = lin;
  p.cin_pad = g.c;
  p.ntaps = g.k;
  p.ntot = g.c;
  p.mrows = lin;
  p.out_shift = 0;
  p.out_valid = (long long)lin * g.c;
  p.div = div;
  p.slope = slope;
  P.x = x;
  P.span = g_knobs.span_ptr ? reinterpret_cast<unsigned long long*>(g_knobs.span_ptr) + 2 * v->tc_launches : nullptr;
  ++v->tc_launches;
  P.trace = (g_knobs.trace_ptr && g_knobs.trace_launch == v->res_launches) ? reinterpret_cast<long long*>(g_knobs.trace_ptr) : nullptr;
  ++v->res_launches;
  const std::string nm = v->convs[v->rb_c1[i][j][0]].name;
  timed_begin(v, st, nm.substr(0, nm.find(".convs1")) + " (whole)", flops);
  const int ctas = g_knobs.max_ctas > 0 ? (int)g_knobs.max_ctas : v->num_sms;
  cudaError_t e = launch_res_tc(P, maps, ctas, st);
  timed_end(v, st);
  if (e != cudaSuccess) return fail(v, L2S_ERR_CUDA, std::string("launch ResBlock ") + nm + ": " + cudaGetErrorString(e));
  return L2S_OK;
}

struct Workspace {
  void* cond;
  void* ma[2];
  float *x, *acc;
  void* xa;
  float* y[L2S_MAX_RK];            // per branch: fp32 residual stream between the steps of a ResBlock
  void *ya[L2S_MAX_RK], *ta[L2S_MAX_RK];   // per branch: activated copies (ping-pong)
  float* spk_vec;
  float* embed;
  int* flags;               // per-item completion counters of the chained ResBlock steps (zeroed at the start of every forward)
  size_t flags_bytes;
  size_t bytes;
};

Workspace carve(const l2s_vocoder* v, int batch, int frames, uint8_t* base) {
  const l2s_config& c = v->cfg;
  const size_t as = act_size(v);
  size_t max_stage = 0;
  long long len = frames;
  for (int i = 0; i < c.n_ups; ++i) {
    len *= c.up_rates[i];
    const size_t e = (size_t)len * v->stage_ch[i];
    if (e > max_stage) max_stage = e;
  }
  const size_t pre_elems = (size_t)frames * c.up_init_ch;
  const size_t ma_elems = max_stage > pre_elems ? max_stage : pre_elems;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    uint8_t* p = base ? base + off : nullptr;
    off += align_up(bytes, 1024);
    return (void*)p;
  };
  Workspace w;
  w.cond = take((size_t)batch * frames * v->convs[v->conv_pre].cin_pad * as);
  w.ma[0] = take((size_t)batch * ma_elems * as);
  w.ma[1] = take((size_t)batch * ma_elems * as);
  w.x = (float*)take((size_t)batch * max_stage * 4);
  w.acc = (float*)take((size_t)batch * max_stage * 4);
  w.xa = take((size_t)batch * max_stage * as);
  for (int j = 0; j < L2S_MAX_RK; ++j) {
    if (j < c.n_rk) {
      w.y[j] = (float*)take((size_t)batch * max_stage * 4);
      w.ya[j] = take((size_t)batch * max_stage * as);
      w.ta[j] = take((size_t)batch * max_stage * as);
    } else { w.y[j] = w.y[0]; w.ya[j] = w.ya[0]; w.ta[j] = w.ta[0]; }
  }
  w.spk_vec = (float*)take((size_t)batch * c.embedding_dim * 4);
  const int units = c.variant == L2S_VARIANT_MULTI_INPUT ? frames / 2 : frames;
  w.embed = (float*)take((size_t)batch * units * c.embedding_dim * 4);
  // one counter per (stage, branch, step, item); an item has at least 100 output rows (128-row tiles minus the c2 halo)
  {
    size_t per_utt = 0;
    long long l2 = frames;
    for (int i = 0; i < c.n_ups; ++i) { l2 *= c.up_rates[i]; per_utt += (size_t)(l2 / 100 + 2); }
    w.flags_bytes = (size_t)batch * per_utt * c.n_rk * c.n_dil * sizeof(int);
    w.flags = (int*)take(w.flags_bytes);
  }
  w.bytes = off;
  return w;
}

// conv_pre, the upsample stages and the MRF stacks: every launch of a forward between the conditioning front end
// and the waveform head.  All buffers live in the workspace, so the sequence can be captured once per
// (batch, frames, workspace) and replayed as a CUDA graph.  *stopped: a debug knob ended the forward early.
int run_chain(l2s_vocoder* v, cudaStream_t st, const Workspace& ws, int batch, int frames, bool* stopped) {
  const l2s_config& c = v->cfg;
  ConvLayer& pre = v->convs[v->conv_pre];
  *stopped = true;
  // chained ResBlock steps (pair_tc.cuh): their per-item counters start at zero in every forward (a memset node in the graph)
  const bool chain_ok = g_knobs.chain && ws.flags && !g_knobs.layer_events && !g_knobs.span_ptr && !g_knobs.trace_ptr && g_knobs.epi_tma == 0;
  if (chain_ok) cudaMemsetAsync(ws.flags, 0, ws.flags_bytes, st);
  size_t flag_off = 0;     // ints handed out so far
  // ---- conv_pre (its consumer applies leaky_relu(0.1): emit the activated copy only)
  int rc = run_conv(v, pre, st, batch, frames, ws.cond, nullptr, ws.ma[0], nullptr, nullptr, 1.f, 0.1f);
  if (rc) return rc;
  v->taps["conv_pre_act"] = {ws.ma[0], (long long)batch * frames * c.up_init_ch, true};
  if (g_knobs.stop_after_pre) return L2S_OK;

  // ---- upsample stages + MRF
  int cur = 0;
  long long len = frames;
  for (int i = 0; i < c.n_ups; ++i) {
    ConvLayer& up = v->convs[v->ups[i]];
    // whole-ResBlock kernels activate the fp32 stream themselves: the upsampler then skips the bf16 copy
    const bool whole = stage_branch_fused(v, i, (int)(len * c.up_rates[i]), batch);
    rc = run_conv(v, up, st, batch, (int)len, ws.ma[cur], ws.x, whole ? nullptr : ws.xa, nullptr, nullptr, 1.f, 0.1f);
    if (rc) return rc;
    len *= c.up_rates[i];
    const int ch = v->stage_ch[i];
    const long long numel = (long long)batch * len * ch;
    const bool last_stage = i == c.n_ups - 1;
    const bool want_raw = last_stage || g_knobs.stop_after_stage == i;
    // A fused step reads its activated input WITH HALO while other CTAs already write the activated
    // output, so fused stages ping-pong the activated buffers (xa -> ya -> ta -> ...); the fp32
    // residual is updated in place (each element is read and written by the same thread).
    if (whole) {
      PkGeom fg;
      bool done = false;
      if (stage_pk_fused(v, i, (int)len, batch, &fg)) {
        // every kernel-size branch of the stage in ONE launch: the branches run back to back on each tile
        rc = run_respk(v, i, 0, c.n_rk, st, batch, (int)len, ws.x, want_raw ? ws.acc : nullptr, last_stage ? nullptr : ws.ma[cur ^ 1],
                       nullptr, ws.acc, (float)c.n_rk, 0.1f);
        if (rc == L2S_OK) done = true;
        else if (rc != L2S_ERR_UNSUPPORTED) return rc;
      }
      // Three tap-by-tap whole-ResBlock branches: the two LARGER kernels (branches 2 and 1) run concurrently on two
      // streams -- the CTAs of one fill the wave-quantisation tail of the other -- each writing its own buffer, and branch 0
      // (the smallest kernel) runs last and adds both: ((x_0 + x_1) + x_2) / 3, bit-identical to the serial chain.
      bool tri = !done && c.n_rk == 3 && g_knobs.narrow_par && !g_res_skew;
      for (int j = 0; tri && j < c.n_rk; ++j) {
        PkGeom pg;
        ResGeom rg;
        if (branch_pk_geom(v, i, j, 1, (int)len, batch, &pg) || !branch_geom(v, i, j, (int)len, batch, &rg)) tri = false;
      }
      if (tri) {
        const bool fork = !g_knobs.layer_events && !g_knobs.span_ptr && !g_knobs.trace_ptr && v->ev_fork;
        cudaStream_t s1 = fork ? v->br_stream[1] : st;
        if (fork) {
          cudaEventRecord(v->ev_fork, st);
          cudaStreamWaitEvent(s1, v->ev_fork, 0);
        }
        rc = run_res(v, i, 2, st, batch, (int)len, ws.x, ws.acc, nullptr, nullptr, 1.f, 0.1f);
        if (rc) return rc;
        rc = run_res(v, i, 1, s1, batch, (int)len, ws.x, ws.y[1], nullptr, nullptr, 1.f, 0.1f);
        if (rc) return rc;
        if (fork) {
          cudaEventRecord(v->ev_join[1], s1);
          cudaStreamWaitEvent(st, v->ev_join[1], 0);
        }
        rc = run_res(v, i, 0, st, batch, (int)len, ws.x, want_raw ? ws.acc : nullptr, last_stage ? nullptr : ws.ma[cur ^ 1], ws.acc,
                     (float)c.n_rk, 0.1f, ws.y[1]);
        if (rc) return rc;
        done = true;
      }
      for (int j = 0; !done && j < c.n_rk; ++j) {
        float* o_raw;
        void* o_act = nullptr;
        const float* a_in = nullptr;
        float dv = 1.f;
        if (j < c.n_rk - 1) { o_raw = ws.acc; a_in = j == 0 ? nullptr : ws.acc; }
        else {
          o_raw = want_raw ? ws.acc : nullptr;
          o_act = last_stage ? nullptr : ws.ma[cur ^ 1];
          a_in = c.n_rk == 1 ? nullptr : ws.acc;
          dv = (float)c.n_rk;
        }
        rc = run_respk(v, i, j, 1, st, batch, (int)len, ws.x, o_raw, o_act, a_in, nullptr, dv, 0.1f);
        if (rc == L2S_ERR_UNSUPPORTED) rc = run_res(v, i, j, st, batch, (int)len, ws.x, o_raw, o_act, a_in, dv, 0.1f);
        if (rc == L2S_ERR_UNSUPPORTED) return fail(v, L2S_ERR_STATE, "whole-ResBlock plan vanished");
        if (rc) return rc;
      }
    }
    bool stage_fused = pairs_fused(v);
    for (int j = 0; stage_fused && j < c.n_rk; ++j)
      for (int m = 0; m < c.n_dil; ++m) {
        const ConvLayer& a1 = v->convs[v->rb_c1[i][j][m]];
        const ConvLayer& a2 = v->convs[v->rb_c2[i][j][m]];
        PairGeom pg;
        if (a1.cin != a1.cout || a1.cin_pad != a1.cin || a1.k != a2.k || a2.dil != 1 ||
            !pair_plan(a1.cin, a1.k, a1.dil, (int)len, batch, (int)g_knobs.pair_smem, g_knobs.dual != 0, g_knobs.cluster != 0, g_knobs.alias_at != 0, false, false, &pg))
          stage_fused = false;
      }
    // Branch-parallel streams: the steps of different branches are independent except that a branch's LAST step adds to the
    // running sum the previous branch's last step wrote.  Branch 0 stays on st, the others fork off it and join back.
    const bool par = !whole && stage_fused && g_knobs.branch_par && c.n_rk > 1 && !g_knobs.layer_events && !g_knobs.span_ptr &&
                     !g_knobs.trace_ptr && v->ev_fork;
    if (par) {
      cudaEventRecord(v->ev_fork, st);
      for (int j = 1; j < c.n_rk; ++j) cudaStreamWaitEvent(v->br_stream[j], v->ev_fork, 0);
    }
    for (int j = 0; !whole && j < c.n_rk; ++j) {
      cudaStream_t sj = (par && j > 0) ? v->br_stream[j] : st;
      const int bj = par ? j : 0;                              // serial: every branch reuses buffer set 0
      // Chain the steps of this branch when they share one item grid (same k: r_out and m_items of every step agree):
      // step m + 1 is launched programmatically and consumes step m item by item (wait_flags / done_flags).
      int chain_items = 0;
      if (chain_ok && stage_fused && c.n_dil > 1) {
        bool same = true;
        PairGeom g0{};
        for (int m = 0; m < c.n_dil && same; ++m) {
          const ConvLayer& a1 = v->convs[v->rb_c1[i][j][m]];
          PairGeom pg;
          if (!pair_plan(a1.cin, a1.k, a1.dil, (int)len, batch, (int)g_knobs.pair_smem, g_knobs.dual != 0, g_knobs.cluster != 0,
                         g_knobs.alias_at != 0, false, false, &pg) || pg.epi_tma)
            same = false;
          else if (m == 0) g0 = pg;
          else if (pg.r_out != g0.r_out || pg.m_items != g0.m_items || pg.total_items != g0.total_items) same = false;
        }
        if (same && (flag_off + (size_t)(c.n_dil - 1) * g0.total_items) * sizeof(int) <= ws.flags_bytes) chain_items = g0.total_items;
      }
      int* step_flags[L2S_MAX_DIL] = {nullptr};
      for (int m = 0; chain_items > 0 && m < c.n_dil - 1; ++m) { step_flags[m] = ws.flags + flag_off; flag_off += (size_t)chain_items; }
      for (int m = 0; m < c.n_dil; ++m) {
        ConvLayer& c1 = v->convs[v->rb_c1[i][j][m]];
        ConvLayer& c2 = v->convs[v->rb_c2[i][j][m]];
        void* act_pp[2] = {ws.ya[bj], ws.ta[bj]};
        const void* in1 = m == 0 ? ws.xa : (stage_fused ? act_pp[(m - 1) & 1] : ws.ya[bj]);
        void* mid_act = stage_fused ? act_pp[m & 1] : ws.ya[bj];     // activated output of a non-final step
        const float* res = m == 0 ? ws.x : ws.y[bj];
        // per (j, m): which outputs the step produces
        float* o_raw;
        void* o_act;
        const float* a_in = nullptr;
        float dv = 1.f;
        if (m < c.n_dil - 1) { o_raw = ws.y[bj]; o_act = mid_act; }
        else if (j < c.n_rk - 1) { o_raw = ws.acc; o_act = nullptr; a_in = j == 0 ? nullptr : ws.acc; }
        else {
          // last branch: mean over branches (true division by num_kernels, models.py:109)
          o_raw = want_raw ? ws.acc : nullptr;
          o_act = last_stage ? nullptr : ws.ma[cur ^ 1];
          a_in = c.n_rk == 1 ? nullptr : ws.acc;
          dv = (float)c.n_rk;
        }
        if (par && m == c.n_dil - 1 && j > 0) cudaStreamWaitEvent(sj, v->ev_acc[j - 1], 0);   // the running sum of the previous branch
        if (stage_fused) {
          // A step that also waits for another stream's event (the running sum of the previous branch) is NOT chained: in a
          // captured graph every incoming edge of a programmatically launched node becomes programmatic, so it would start
          // before that branch has finished, and the running sum is not covered by the item counters.
          const bool ev_dep = par && m == c.n_dil - 1 && j > 0;
          rc = run_pair(v, c1, c2, sj, batch, (int)len, in1, res, o_raw, o_act, a_in, dv, 0.1f,
                        (chain_items > 0 && m > 0 && !ev_dep) ? step_flags[m - 1] : nullptr,
                        (chain_items > 0 && m < c.n_dil - 1) ? step_flags[m] : nullptr);
          if (rc == L2S_ERR_UNSUPPORTED) return fail(v, L2S_ERR_STATE, "fused plan vanished for " + c1.name);
        } else {
          rc = run_conv(v, c1, sj, batch, (int)len, in1, nullptr, ws.ta[bj], nullptr, nullptr, 1.f, 0.1f);
          if (rc) return rc;
          rc = run_conv(v, c2, sj, batch, (int)len, ws.ta[bj], o_raw, o_act, res, a_in, dv, 0.1f);
        }
        if (rc) return rc;
        if (par && m == c.n_dil - 1 && j < c.n_rk - 1) cudaEventRecord(v->ev_acc[j], sj);
      }
    }
    if (par)
      for (int j = 1; j < c.n_rk; ++j) {
        cudaEventRecord(v->ev_join[j], v->br_stream[j]);
        cudaStreamWaitEvent(st, v->ev_join[j], 0);
      }
    cur ^= 1;
    if (g_knobs.stop_after_stage == i) {
      v->taps["ups"] = {ws.x, numel, false};
      v->taps["mrf"] = {ws.acc, numel, false};
      return L2S_OK;
    }
  }

  *stopped = false;
  return L2S_OK;
}

int forward_impl(l2s_vocoder* v, void* stream, const int64_t* code, const void* mel, int32_t mel_dtype, const void* spkr,
                 int32_t batch, int32_t units, int32_t frames, float* out, int16_t* out_i16, void* workspace,
                 int64_t workspace_bytes) {
  if (!v) return L2S_ERR_INVALID;
  std::shared_lock<std::shared_mutex> knobs(g_knob_mu);
  std::lock_guard<std::mutex> lock(v->mu);
  if (!v->finalized) return fail(v, L2S_ERR_STATE, "l2s_finalize has not been called");
  if (v->err_host && *(volatile int*)v->err_host) {
    // An EARLIER forward on this handle clamped an out-of-range id (the reference raises IndexError on the CPU and
    // device-asserts on CUDA): report it now, late rather than never, without synchronising.  This call does no work.
    const int f = *(volatile int*)v->err_host;
    *(volatile int*)v->err_host = 0;
    return fail(v, L2S_ERR_INDEX, (f & 1) ? "index out of range in self (a unit id outside the dict table, seen by an earlier forward)"
                                          : "index out of range in self (a speaker id outside the table, seen by an earlier forward)");
  }
  const l2s_config& c = v->cfg;
  const bool multi = c.variant == L2S_VARIANT_MULTI_INPUT;
  if (batch < 1 || units < 1 || frames < 1) return fail(v, L2S_ERR_SHAPE, "empty batch / sequence");
  if (!code || (!out && !out_i16) || !workspace) return fail(v, L2S_ERR_INVALID, "null pointer");
  if (multi) {
    if (!mel) return fail(v, L2S_ERR_INVALID, "mel is required (models_multi_input.py:65)");
    if (frames != 2 * units) {
      char b[160];
      snprintf(b, sizeof b, "Sizes of tensors must match except in dimension 1. Expected size %d but got size %d (mel frames vs 2*units)",
               frames, 2 * units);
      return fail(v, L2S_ERR_SHAPE, b);
    }
    if (mel_dtype < 0 || mel_dtype > 2) return fail(v, L2S_ERR_INVALID, "mel dtype");
  } else if (frames != units) {
    return fail(v, L2S_ERR_SHAPE, "unit-only variant: frames must equal units");
  }
  if (c.multispkr && !spkr) return fail(v, L2S_ERR_INVALID, "spkr is required");
  if ((uintptr_t)workspace % 256 != 0) return fail(v, L2S_ERR_WORKSPACE, "workspace must be 256-byte aligned");
  Workspace ws = carve(v, batch, frames, (uint8_t*)workspace);
  if ((int64_t)ws.bytes > workspace_bytes) return fail(v, L2S_ERR_WORKSPACE, "workspace too small");
  int dev_now = -1;
  cudaGetDevice(&dev_now);
  if (dev_now != v->device) cudaSetDevice(v->device);
  cudaStream_t st = (cudaStream_t)stream;
  const bool bf = is_bf16(v);
  const int E = c.embedding_dim;
  v->taps.clear();
  v->timed_used = 0;
  v->pair_launches = 0;
  v->res_launches = 0;
  v->tc_launches = 0;
  cudaError_t e;
  ConvLayer& pre = v->convs[v->conv_pre];

  // ---- conditioning front end
  timed_begin(v, st, "front_end", 0.0);
  float* embed_tap = g_knobs.embed_tap ? ws.embed : nullptr;
  if (multi) {
    // the speaker projection runs inside the conditioning kernel (every block projects its utterance's embedding: one launch
    // and one kernel boundary less in front of conv_pre); knob front_fuse = 0 or an oversized spk_dim: the separate kernel
    const bool spk_in_block = c.multispkr && g_knobs.front_fuse && c.spk_dim <= kCondMaxSpk;
    if (c.multispkr && !spk_in_block) {
      spk_project_kernel<<<batch, 512, c.spk_dim * sizeof(float), st>>>((const float*)spkr, v->d_spk_w, v->d_spk_b, ws.spk_vec,
                                                                        c.spk_dim, E);
    }
    CondParams cp{};
    if (spk_in_block) { cp.spk_raw = (const float*)spkr; cp.spk_w = v->d_spk_w; cp.spk_b = v->d_spk_b; cp.spk_dim = c.spk_dim; }
    cp.code = (const long long*)code;
    cp.mel = mel;
    cp.mel_dtype = mel_dtype;
    cp.spk_vec = ws.spk_vec;
    cp.dict = v->d_dict;
    cp.wt = v->d_wt;
    cp.tab = v->d_unit_tab;
    cp.wt_bias = v->d_wt_b;
    cp.fc_t = v->d_fc_t;
    cp.fc_bias = v->d_fc_b;
    cp.cond = ws.cond;
    cp.embed_tap = embed_tap;
    cp.err_flag = v->err_dev;
    cp.batch = batch; cp.units = units; cp.frames = frames; cp.e = E; cp.num_mels = c.num_mels;
    cp.num_embeddings = c.num_embeddings; cp.cin_pad = pre.cin_pad; cp.has_spk = c.multispkr ? 1 : 0;
    dim3 grid((frames + kCondFrames * kCondPasses - 1) / (kCondFrames * kCondPasses), batch);
    if (bf) cond_multi_kernel<__nv_bfloat16><<<grid, kCondThreads, 0, st>>>(cp);
    else cond_multi_kernel<float><<<grid, kCondThreads, 0, st>>>(cp);
  } else {
    CondUnitParams cp{};
    cp.code = (const long long*)code;
    cp.spk_id = (const long long*)spkr;
    cp.dict = v->d_dict;
    cp.spk_table = v->d_spk_w;
    cp.cond = ws.cond;
    cp.embed_tap = embed_tap;
    cp.err_flag = v->err_dev;
    cp.batch = batch; cp.units = units; cp.e = E; cp.num_embeddings = c.num_embeddings;
    cp.num_speakers = c.num_speakers; cp.cin_pad = pre.cin_pad; cp.has_spk = c.multispkr ? 1 : 0;
    dim3 grid(units, batch);
    if (bf) cond_unit_kernel<__nv_bfloat16><<<grid, 128, 0, st>>>(cp);
    else cond_unit_kernel<float><<<grid, 128, 0, st>>>(cp);
  }
  timed_end(v, st);
  if ((e = cudaGetLastError()) != cudaSuccess) return fail(v, L2S_ERR_CUDA, std::string("front end: ") + cudaGetErrorString(e));
  v->taps["cond"] = {ws.cond, (long long)batch * frames * pre.cin_pad, true};
  if (embed_tap) v->taps["embed"] = {ws.embed, (long long)batch * units * E, false};

  // ---- conv_pre, upsample stages, MRF stacks: eager, or replayed from a captured CUDA graph
  {
    const bool debug_run = g_knobs.stop_after_pre || g_knobs.stop_after_stage >= 0 || g_knobs.layer_events || g_knobs.span_ptr ||
                           g_knobs.trace_ptr;
    const bool graph_ok = g_knobs.use_graph && !debug_run && v->cfg.precision != L2S_PREC_FP32;
    bool stopped = false;
    int rc = L2S_OK;
    l2s_vocoder::ChainGraph* slot = nullptr;
    if (graph_ok) {
      for (auto& gph : v->graphs)
        if (gph.batch == batch && gph.frames == frames && gph.workspace == workspace && gph.epoch == g_knobs.epoch) slot = &gph;
      if (!slot) {
        if (v->graphs.size() >= 16) {   // keep the cache small: drop everything (shapes rarely vary that much)
          for (auto& gph : v->graphs) if (gph.exec) cudaGraphExecDestroy(gph.exec);
          v->graphs.clear();
        }
        v->graphs.push_back({batch, frames, workspace, g_knobs.epoch, 0, nullptr});
        slot = &v->graphs.back();
      }
    }
    if (slot && slot->exec) {
      if ((e = cudaGraphLaunch(slot->exec, st)) != cudaSuccess)
        return fail(v, L2S_ERR_CUDA, std::string("cudaGraphLaunch: ") + cudaGetErrorString(e));
    } else if (slot && slot->seen >= 1) {
      // second forward with this shape: capture on the internal stream (the caller's may be the legacy default
      // stream, which cannot be captured), then replay on the caller's stream
      if (!v->capture_stream && (e = cudaStreamCreateWithFlags(&v->capture_stream, cudaStreamNonBlocking)) != cudaSuccess)
        return fail(v, L2S_ERR_CUDA, std::string("cudaStreamCreate: ") + cudaGetErrorString(e));
      cudaGraph_t graph = nullptr;
      if ((e = cudaStreamBeginCapture(v->capture_stream, cudaStreamCaptureModeThreadLocal)) != cudaSuccess)
        return fail(v, L2S_ERR_CUDA, std::string("cudaStreamBeginCapture: ") + cudaGetErrorString(e));
      rc = run_chain(v, v->capture_stream, ws, batch, frames, &stopped);
      e = cudaStreamEndCapture(v->capture_stream, &graph);
      if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
      if (e != cudaSuccess || !graph) return fail(v, L2S_ERR_CUDA, std::string("cudaStreamEndCapture: ") + cudaGetErrorString(e));
      e = cudaGraphInstantiate(&slot->exec, graph, 0);
      cudaGraphDestroy(graph);
      if (e != cudaSuccess) { slot->exec = nullptr; return fail(v, L2S_ERR_CUDA, std::string("cudaGraphInstantiate: ") + cudaGetErrorString(e)); }
      if ((e = cudaGraphLaunch(slot->exec, st)) != cudaSuccess)
        return fail(v, L2S_ERR_CUDA, std::string("cudaGraphLaunch: ") + cudaGetErrorString(e));
    } else {
      rc = run_chain(v, st, ws, batch, frames, &stopped);   // eager (first use of a shape, debug runs, fp32 mode)
      if (rc) return rc;
      if (slot) ++slot->seen;
      if (stopped) return L2S_OK;
    }
  }
  long long len = (long long)frames * hop_of(c);

  // ---- waveform head
  PostParams pp{};
  pp.in = ws.acc;
  for (size_t i = 0; i < v->post_w_host.size() && i < sizeof(pp.wc) / sizeof(float); ++i) pp.wc[i] = v->post_w_host[i];
  pp.bias = v->post_bias;
  pp.out = out;
  pp.out_i16 = out_i16;
  pp.batch = batch;
  pp.len = (int)len;
  pp.c = v->stage_ch.back();
  dim3 grid((unsigned)((len + kPostTile - 1) / kPostTile), batch);
  timed_begin(v, st, "conv_post", 2.0 * pp.c * 7 * (double)batch * len);
  const dim3 grid_rows((unsigned)((len + kPostRowsOut - 1) / kPostRowsOut), batch);
  if (pp.c == 16 && g_knobs.post_rows) post_rows_kernel<16><<<grid_rows, kPostTile, 0, st>>>(pp);
  else if (pp.c == 32 && g_knobs.post_rows) post_rows_kernel<32><<<grid_rows, kPostTile, 0, st>>>(pp);
  else if (pp.c == 16) post_kernel<16><<<grid, kPostTile, (kPostTile + 6) * post_pitch(pp.c) * sizeof(float), st>>>(pp);
  else if (pp.c == 32) post_kernel<32><<<grid, kPostTile, (kPostTile + 6) * post_pitch(pp.c) * sizeof(float), st>>>(pp);
  else {
    // C = 48 / 64: the staged tile ((kPostTile + 6) rows of C + 4 floats, 71 KB at C = 64) is larger than the 48 KB of
    // dynamic shared memory a launch gets without opting in
    static bool configured[64] = {false};
    if (v->device >= 0 && v->device < 64 && !configured[v->device]) {
      if ((e = cudaFuncSetAttribute(post_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)((kPostTile + 6) * post_pitch(kPostMaxC) * sizeof(float)))) != cudaSuccess)
        return fail(v, L2S_ERR_CUDA, std::string("post: ") + cudaGetErrorString(e));
      configured[v->device] = true;
    }
    post_kernel<0><<<grid, kPostTile, (kPostTile + 6) * post_pitch(pp.c) * sizeof(float), st>>>(pp);
  }
  timed_end(v, st);
  if ((e = cudaGetLastError()) != cudaSuccess) return fail(v, L2S_ERR_CUDA, std::string("post: ") + cudaGetErrorString(e));
  return L2S_OK;
}

}  // namespace

// ------------------------------------------------------------------ C ABI

extern "C" {

int l2s_create(const l2s_config* cfg, l2s_vocoder** out) {
  if (!cfg || !out) return L2S_ERR_INVALID;
  l2s_vocoder* v = new (std::nothrow) l2s_vocoder();
  if (!v) return L2S_ERR_INVALID;
  v->cfg = *cfg;
  const int rc = build_layers(v);
  *out = v;   // returned even on failure so the caller can read l2s_last_error, then destroy
  return rc;
}

void l2s_destroy(l2s_vocoder* v) {
  if (!v) return;
  if (v->finalized) {
    int dev = -1;
    cudaGetDevice(&dev);
    if (dev != v->device) cudaSetDevice(v->device);
    for (auto& gph : v->graphs) if (gph.exec) cudaGraphExecDestroy(gph.exec);
    if (v->capture_stream) cudaStreamDestroy(v->capture_stream);
    for (int j = 0; j < L2S_MAX_RK; ++j) {
      if (v->br_stream[j]) cudaStreamDestroy(v->br_stream[j]);
      if (v->ev_acc[j]) cudaEventDestroy(v->ev_acc[j]);
      if (v->ev_join[j]) cudaEventDestroy(v->ev_join[j]);
    }
    if (v->ev_fork) cudaEventDestroy(v->ev_fork);
    for (void* p : v->dev_allocs) cudaFree(p);
    if (v->err_host) cudaFreeHost(v->err_host);
    if (dev >= 0 && dev != v->device) cudaSetDevice(dev);
  }
  delete v;
}

int l2s_set_weight(l2s_vocoder* v, const char* name, const float* host_data, int64_t numel) {
  if (!v || !name || !host_data) return L2S_ERR_INVALID;
  std::lock_guard<std::mutex> lock(v->mu);
  if (v->finalized) return fail(v, L2S_ERR_STATE, "weights are frozen after l2s_finalize");
  auto it = v->expected.find(name);
  if (it == v->expected.end()) return fail(v, L2S_ERR_INVALID, std::string("unexpected weight name: ") + name);
  if (it->second != numel) {
    char b[160];
    snprintf(b, sizeof b, "size mismatch for %s: expected %lld elements, got %lld", name, it->second, (long long)numel);
    return fail(v, L2S_ERR_SHAPE, b);
  }
  v->weights[name].assign(host_data, host_data + numel);
  return L2S_OK;
}

int l2s_finalize(l2s_vocoder* v, int device) {
  if (!v) return L2S_ERR_INVALID;
  std::lock_guard<std::mutex> lock(v->mu);
  if (v->finalized) return fail(v, L2S_ERR_STATE, "already finalized");
  for (auto& kv : v->expected)
    if (!v->weights.count(kv.first)) return fail(v, L2S_ERR_STATE, "missing weight: " + kv.first);
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev < 1) return fail(v, L2S_ERR_CUDA, "no CUDA device: this library has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(v, L2S_ERR_INVALID, "bad device index");
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return fail(v, L2S_ERR_CUDA, cudaGetErrorString(e));
  if (prop.major != 10) {
    char b[128];
    snprintf(b, sizeof b, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
    return fail(v, L2S_ERR_UNSUPPORTED, b);
  }
  int prev = -1;
  cudaGetDevice(&prev);
  if ((e = cudaSetDevice(device)) != cudaSuccess) return fail(v, L2S_ERR_CUDA, cudaGetErrorString(e));
  v->device = device;
  v->num_sms = prop.multiProcessorCount;
  const l2s_config& c = v->cfg;
  const bool bf = is_bf16(v);
  const int E = c.embedding_dim;

  for (ConvLayer& L : v->convs) {
    std::vector<float> pw, pb;
    pack_conv(L, v->weights[L.name + ".weight"], v->weights[L.name + ".bias"], &pw, &pb);
    if (bf) {
      std::vector<uint16_t> hw(pw.size());
      for (size_t i = 0; i < pw.size(); ++i) hw[i] = f2bf(pw[i]);
      L.w_dev = dev_upload<uint16_t>(v, hw.data(), hw.size(), &e);
    } else {
      if (is_tf32(v))
        for (float& x : pw) x = f2tf32(x);   // the tensor core would truncate; round to nearest instead
      L.w_dev = dev_upload<float>(v, pw.data(), pw.size(), &e);
    }
    if (e != cudaSuccess) return fail(v, L2S_ERR_CUDA, std::string("upload ") + L.name + ": " + cudaGetErrorString(e));
    L.bias_dev = dev_upload<float>(v, pb.data(), pb.size(), &e);
    if (e != cudaSuccess) return fail(v, L2S_ERR_CUDA, cudaGetErrorString(e));
  }
  {
    const std::vector<float> zeros(256, 0.f);
    v->d_zero_bias = dev_upload<float>(v, zeros.data(), zeros.size(), &e);
    if (e != cudaSuccess) return fail(v, L2S_ERR_CUDA, cudaGetErrorString(e));
  }
  // time-packed whole-ResBlock kernel: block-Toeplitz weights and per-column bias constants of the C <= 64 stages
  v->pk_bias.assign((size_t)c.n_ups, std::vector<float*>((size_t)c.n_rk, nullptr));
  v->pk_bias_stage.assign((size_t)c.n_ups, nullptr);
  v->pk_bias_host.assign((size_t)c.n_ups, std::vector<std::vector<float>>((size_t)c.n_rk));
  for (int i = 0; i < c.n_ups; ++i) {
    const int ch = v->stage_ch[i];
    if (!v->pk_ok[i]) continue;
    std::vector<float> stage_cols;
    for (int j = 0; j < c.n_rk; ++j) {
      std::vector<float> cols((size_t)kPkBiasRows * 128, 0.f), run((size_t)ch, 0.f);
      for (int m = 0; m < c.n_dil; ++m) {
        for (int which = 0; which < 2; ++which) {
          ConvLayer& L = v->convs[which ? v->rb_c2[i][j][m] : v->rb_c1[i][j][m]];
          std::vector<float> pk;
          pk_pack_weights(v->weights[L.name + ".weight"].data(), ch, L.k, &pk);
          std::vector<uint16_t> hw(pk.size());
          for (size_t q = 0; q < pk.size(); ++q) hw[q] = f2bf(pk[q]);
          L.wpk_dev = dev_upload<uint16_t>(v, hw.data(), hw.size(), &e);
          if (e != cudaSuccess) return fail(v, L2S_ERR_CUDA, std::string("upload packed ") + L.name + ": " + cudaGetErrorString(e));
          L.pk_groups = (int)(pk.size() / (128 * 64));
          const std::vector<float>& b = v->weights[L.name + ".bias"];
          if (which) for (int q = 0; q < ch; ++q) run[q] += b[q];            // running sum of the c2 biases
          for (int col = 0; col < 128; ++col) cols[(size_t)(2 * m + which) * 128 + col] = which ? run[col % ch] : b[col % ch];
        }
      }
      for (int col = 0; col < 128; ++col) cols[(size_t)(2 * kPkMaxDil) * 128 + col] = run[col % ch];   // output epilogue: all c2 biases
      v->pk_bias[i][j] = dev_upload<float>(v, cols.data(), cols.size(), &e);
      if (e != cudaSuccess) return fail(v, L2S_ERR_CUDA, cudaGetErrorString(e));
      stage_cols.insert(stage_cols.end(), cols.begin(), cols.end());
      std::vector<float>& hb = v->pk_bias_host[i][j];
      hb.assign((size_t)kPkBiasRows * 64, 0.f);
      for (int row = 0; row < kPkBiasRows; ++row)
        for (int q = 0; q < ch; ++q) hb[(size_t)row * 64 + q] = cols[(size_t)row * 128 + q];
    }
    v->pk_bias_stage[i] = dev_upload<float>(v, stage_cols.data(), stage_cols.size(), &e);
    if (e != cudaSuccess) return fail(v, L2S_ERR_CUDA, cudaGetErrorString(e));
  }
  {
    const std::vector<float>& d = v->weights["dict.weight"];
    v->d_dict = dev_upload<float>(v, d.data(), d.size(), &e);
    if (e != cudaSuccess) return fail(v, L2S_ERR_CUDA, cudaGetErrorString(e));
  }
  if (c.variant == L2S_VARIANT_MULTI_INPUT) {
    // unit ConvTranspose1d weight (E_in, E_out, 4) -> [4][E_in][E_out]
    const std::vector<float>& w = v->weights["layer.0.weight"];
    std::vector<float> wt((size_t)4 * E * E);
    for (int ci = 0; ci < E; ++ci)
      for (int co = 0; co < E; ++co)
        for (int j = 0; j < 4; ++j) wt[((size_t)j * E + ci) * E + co] = w[((size_t)ci * E + co) * 4 + j];
    v->d_wt = dev_upload<float>(v, wt.data(), wt.size(), &e);
    if (e != cudaSuccess) return fail(v, L2S_ERR_CUDA, cudaGetErrorString(e));
    v->d_wt_b = dev_upload<float>(v, v->weights["layer.0.bias"].data(), E, &e);
    {
      // tab[j][id][co] = sum_ci dict[id][ci] * W[ci][co][j], accumulated in double and rounded once
      const std::vector<float>& d = v->weights["dict.weight"];
      const int n_emb = c.num_embeddings;
      std::vector<float> tab((size_t)4 * n_emb * E);
      std::vector<double> acc((size_t)E);
      for (int j = 0; j < 4; ++j)
        for (int id = 0; id < n_emb; ++id) {
          std::fill(acc.begin(), acc.end(), 0.0);
          for (int ci = 0; ci < E; ++ci) {
            const double x = d[(size_t)id * E + ci];
            const float* wrow = &wt[((size_t)j * E + ci) * E];
            for (int co = 0; co < E; ++co) acc[co] += x * (double)wrow[co];
          }
          for (int co = 0; co < E; ++co) tab[((size_t)j * n_emb + id) * E + co] = (float)acc[co];
        }
      v->d_unit_tab = dev_upload<float>(v, tab.data(), tab.size(), &e);
      if (e != cudaSuccess) return fail(v, L2S_ERR_CUDA, cudaGetErrorString(e));
    }
    const std::vector<float>& fw = v->weights["fc.weight"];   // (out, in)
    std::vector<float> ft((size_t)E * E);
    for (int o = 0; o < E; ++o)
      for (int k = 0; k < E; ++k) ft[(size_t)k * E + o] = fw[(size_t)o * E + k];
    v->d_fc_t = dev_upload<float>(v, ft.data(), ft.size(), &e);
    v->d_fc_b = dev_upload<float>(v, v->weights["fc.bias"].data(), E, &e);
    if (c.multispkr) {
      v->d_spk_w = dev_upload<float>(v, v->weights["spkr.weight"].data(), v->weights["spkr.weight"].size(), &e);
      v->d_spk_b = dev_upload<float>(v, v->weights["spkr.bias"].data(), E, &e);
    }
    if (e != cudaSuccess) return fail(v, L2S_ERR_CUDA, cudaGetErrorString(e));
  } else if (c.multispkr) {
    v->d_spk_w = dev_upload<float>(v, v->weights["spkr.weight"].data(), v->weights["spkr.weight"].size(), &e);
    if (e != cudaSuccess) return fail(v, L2S_ERR_CUDA, cudaGetErrorString(e));
  }
  {
    // conv_post weight (1, C, 7) -> [7][C]
    const int C = v->stage_ch.back();
    const std::vector<float>& w = v->weights["conv_post.weight"];
    std::vector<float> pw((size_t)7 * C);
    for (int ch = 0; ch < C; ++ch)
      for (int j = 0; j < 7; ++j) pw[(size_t)j * C + ch] = w[(size_t)ch * 7 + j];
    v->d_post_w = dev_upload<float>(v, pw.data(), pw.size(), &e);
    v->post_w_host = pw;
    if (e != cudaSuccess) return fail(v, L2S_ERR_CUDA, cudaGetErrorString(e));
    v->post_bias = v->weights["conv_post.bias"][0];
  }
  for (int j = 1; j < c.n_rk && j < L2S_MAX_RK; ++j) {
    if ((e = cudaStreamCreateWithFlags(&v->br_stream[j], cudaStreamNonBlocking)) != cudaSuccess) return fail(v, L2S_ERR_CUDA, cudaGetErrorString(e));
    cudaEventCreateWithFlags(&v->ev_join[j], cudaEventDisableTiming);
  }
  for (int j = 0; j < L2S_MAX_RK; ++j) cudaEventCreateWithFlags(&v->ev_acc[j], cudaEventDisableTiming);
  if ((e = cudaEventCreateWithFlags(&v->ev_fork, cudaEventDisableTiming)) != cudaSuccess) return fail(v, L2S_ERR_CUDA, cudaGetErrorString(e));
  if ((e = cudaHostAlloc((void**)&v->err_host, sizeof(int), cudaHostAllocMapped)) != cudaSuccess)
    return fail(v, L2S_ERR_CUDA, cudaGetErrorString(e));
  *v->err_host = 0;
  if ((e = cudaHostGetDevicePointer((void**)&v->err_dev, v->err_host, 0)) != cudaSuccess)
    return fail(v, L2S_ERR_CUDA, cudaGetErrorString(e));
  if ((e = cudaDeviceSynchronize()) != cudaSuccess) return fail(v, L2S_ERR_CUDA, cudaGetErrorString(e));
  v->weights.clear();
  v->finalized = true;
  if (prev >= 0 && prev != device) cudaSetDevice(prev);
  return L2S_OK;
}

int64_t l2s_workspace_bytes(l2s_vocoder* v, int32_t batch, int32_t frames) {
  if (!v || batch < 1 || frames < 1 || v->convs.empty()) return -1;
  return (int64_t)carve(v, batch, frames, nullptr).bytes;
}

int32_t l2s_hop(l2s_vocoder* v) { return v ? hop_of(v->cfg) : -1; }

int l2s_forward(l2s_vocoder* v, void* stream, const int64_t* code, const void* mel, int32_t mel_dtype, const void* spkr,
                int32_t batch, int32_t units, int32_t frames, float* out, void* workspace, int64_t workspace_bytes) {
  return forward_impl(v, stream, code, mel, mel_dtype, spkr, batch, units, frames, out, nullptr, workspace, workspace_bytes);
}

int l2s_forward_i16(l2s_vocoder* v, void* stream, const int64_t* code, const void* mel, int32_t mel_dtype, const void* spkr,
                    int32_t batch, int32_t units, int32_t frames, float* out, int16_t* out_i16, void* workspace,
                    int64_t workspace_bytes) {
  if (!out_i16) return fail(v, L2S_ERR_INVALID, "out_i16 is null");
  return forward_impl(v, stream, code, mel, mel_dtype, spkr, batch, units, frames, out, out_i16, workspace, workspace_bytes);
}

int l2s_poll_index_error(l2s_vocoder* v) {
  if (!v || !v->err_host) return L2S_ERR_STATE;
  const int f = *(volatile int*)v->err_host;
  *(volatile int*)v->err_host = 0;
  if (f) return fail(v, L2S_ERR_INDEX, (f & 1) ? "index out of range in self (unit id outside the dict table)"
                                                : "index out of range in self (speaker id outside the table)");
  return L2S_OK;
}

int32_t l2s_launch_count(l2s_vocoder* v, int32_t batch, int32_t frames) {
  if (!v) return -1;
  std::shared_lock<std::shared_mutex> knobs(g_knob_mu);
  const l2s_config& c = v->cfg;
  int n = (int)v->convs.size() + 1 /* post */ + 1 /* cond */;
  if (pairs_fused(v)) n -= c.n_ups * c.n_rk * c.n_dil;   // one launch per (c1, c2) step
  long long len = frames;
  for (int i = 0; i < c.n_ups; ++i) {
    len *= c.up_rates[i];
    if (batch > 0 && frames > 0 && stage_branch_fused(v, i, (int)len, batch)) {
      n -= c.n_rk * (c.n_dil - 1);   // one per ResBlock
      PkGeom fg;
      if (stage_pk_fused(v, i, (int)len, batch, &fg)) n -= c.n_rk - 1;   // one per stage
    }
  }
  if (c.variant == L2S_VARIANT_MULTI_INPUT && c.multispkr && !(g_knobs.front_fuse && c.spk_dim <= kCondMaxSpk)) n += 1;   // separate speaker projection
  return n;
}

const char* l2s_last_error(l2s_vocoder* v) { return v ? v->err.c_str() : "null handle"; }
const char* l2s_version(void) { return "l2s_vocoder 0.2 (sm_100a)"; }

int l2s_debug_tap(l2s_vocoder* v, const char* name, float* host_dst, int64_t numel) {
  if (!v || !name || !host_dst) return L2S_ERR_INVALID;
  std::lock_guard<std::mutex> lock(v->mu);
  auto it = v->taps.find(name);
  if (it == v->taps.end()) return fail(v, L2S_ERR_INVALID, std::string("no such tap: ") + name);
  if (it->second.numel != numel) {
    char b[128];
    snprintf(b, sizeof b, "tap %s has %lld elements, caller asked for %lld", name, it->second.numel, (long long)numel);
    return fail(v, L2S_ERR_SHAPE, b);
  }
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) return fail(v, L2S_ERR_CUDA, cudaGetErrorString(e));
  if (it->second.act && is_bf16(v)) {
    std::vector<uint16_t> tmp((size_t)numel);
    e = cudaMemcpy(tmp.data(), it->second.ptr, (size_t)numel * 2, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return fail(v, L2S_ERR_CUDA, cudaGetErrorString(e));
    for (int64_t i = 0; i < numel; ++i) {
      const uint32_t u = (uint32_t)tmp[(size_t)i] << 16;
      memcpy(&host_dst[i], &u, 4);
    }
  } else {
    e = cudaMemcpy(host_dst, it->second.ptr, (size_t)numel * 4, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return fail(v, L2S_ERR_CUDA, cudaGetErrorString(e));
  }
  return L2S_OK;
}

int l2s_debug_conv(const l2s_conv_desc* d, int32_t impl, int32_t device, void* stream, char* err, int32_t err_len) {
  auto say = [&](const char* m) {
    if (err && err_len > 0) snprintf(err, (size_t)err_len, "%s", m);
  };
  if (!d) { say("null desc"); return L2S_ERR_INVALID; }
  std::shared_lock<std::shared_mutex> knobs(g_knob_mu);
  if (d->ntaps < 1 || d->ntaps > kMaxTaps) { say("ntaps"); return L2S_ERR_INVALID; }
  cudaError_t e = cudaSetDevice(device);
  if (e != cudaSuccess) { say(cudaGetErrorString(e)); return L2S_ERR_CUDA; }
  ConvParams p{};
  p.in = d->in; p.w = d->w; p.bias = d->bias; p.out_raw = d->out_raw; p.out_act = d->out_act; p.res = d->res;
  p.acc_in = d->acc_in;
  p.batch = d->batch; p.lin = d->lin; p.cin_pad = d->cin_pad; p.ntaps = d->ntaps; p.ntot = d->ntot; p.mrows = d->mrows;
  for (int j = 0; j < d->ntaps; ++j) p.tap_off[j] = d->tap_off[j];
  p.out_shift = d->out_shift; p.out_valid = d->out_valid;
  p.div = d->scale; p.slope = d->slope;
  cudaStream_t st = (cudaStream_t)stream;
  if (impl == 0) {
    e = d->act_bf16 ? launch_conv_simt<__nv_bfloat16>(p, st) : launch_conv_simt<float>(p, st);
  } else {
    p.act_f32 = d->act_bf16 ? 0 : 1;   // fp32 operands run as kind::tf32
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    TcTune tune = current_tune(nullptr);
    if (g_knobs.max_ctas <= 0) tune.max_ctas = sms;
    if (impl == 2) { say("impl 2 (descriptor base-offset probe) was removed: it gives wrong results on sm_100a"); return L2S_ERR_UNSUPPORTED; }
    if (impl == 3) tune.per_tap = 1;
    TcGeom g;
    if (!tc_plan(p, d->batch, tune, &g)) { say("no tcgen05 plan"); return L2S_ERR_UNSUPPORTED; }
    CUtensorMap tmA, tmW;
    if (!make_tmap_3d(&tmW, d->w, g.esz, (uint64_t)d->cin_pad, (uint64_t)d->ntot, (uint64_t)d->ntaps,
                      (uint32_t)(g.rb / g.esz), (uint32_t)(g.cg2 ? g.nt / 2 : g.nt), (uint32_t)g.tb) ||
        !make_tmap_3d(&tmA, d->in, g.esz, (uint64_t)d->cin_pad, (uint64_t)d->lin, (uint64_t)d->batch,
                      (uint32_t)(g.rb / g.esz), (uint32_t)g.box_rows, 1u)) {
      say("cuTensorMapEncodeTiled failed");
      return L2S_ERR_CUDA;
    }
    e = launch_conv_tc(p, g, tmA, tmW, tune.max_ctas, st, reinterpret_cast<long long*>(g_knobs.trace_ptr));
    if (e == cudaSuccess && err && err_len > 0 && g_knobs.plan_report) {
      snprintf(err, (size_t)err_len, "plan msub=%d nt=%d kc=%d tb=%d sa=%d sb=%d smem=%d tmem=%d items=%d ctas_per_sm=%d",
               g.msub, g.nt, g.kc, g.tb, g.sa, g.sb, g.smem_bytes, g.tmem_cols, g.total_items, g.ctas_per_sm);
    }
  }
  if (e != cudaSuccess) { say(cudaGetErrorString(e)); return L2S_ERR_CUDA; }
  return L2S_OK;
}

int l2s_debug_layer_time(l2s_vocoder* v, int32_t idx, float* ms, double* flops, char* name, int32_t name_len) {
  if (!v || !ms) return L2S_ERR_INVALID;
  std::lock_guard<std::mutex> lock(v->mu);
  if (idx < 0 || (size_t)idx >= v->timed_used) return L2S_ERR_INVALID;
  l2s_vocoder::Timed& t = v->timed[(size_t)idx];
  cudaError_t e = cudaEventSynchronize(t.b);
  if (e == cudaSuccess) e = cudaEventElapsedTime(ms, t.a, t.b);
  if (e != cudaSuccess) return fail(v, L2S_ERR_CUDA, cudaGetErrorString(e));
  if (flops) *flops = t.flops;
  if (name && name_len > 0) snprintf(name, (size_t)name_len, "%s", t.name.c_str());
  return L2S_OK;
}

int l2s_debug_set(const char* key, int64_t value) {
  if (!key) return L2S_ERR_INVALID;
  std::unique_lock<std::shared_mutex> knobs(g_knob_mu);
  const std::string k(key);
  ++g_knobs.epoch;
  if (k == "use_graph") { g_knobs.use_graph = value; return L2S_OK; }
  if (k == "force_simt") g_knobs.force_simt = value;
  else if (k == "stop_after_stage") g_knobs.stop_after_stage = value;
  else if (k == "stop_after_pre") g_knobs.stop_after_pre = value;
  else if (k == "per_tap") g_knobs.per_tap = value;
  else if (k == "sa_min") g_knobs.sa_min = value;
  else if (k == "dual") g_knobs.dual = value;
  else if (k == "fuse_pairs") g_knobs.fuse_pairs = value;
  else if (k == "fuse_branch") g_knobs.fuse_branch = value;
  else if (k == "res_mode") g_knobs.res_mode = value;
  else if (k == "res_msub") g_knobs.res_msub = value;
  else if (k == "res_single_pct") g_res_single_pct = (int)value;
  else if (k == "res_quad_pct") g_res_quad_pct = (int)value;
  else if (k == "res_cg2") g_res_cg2 = (int)value;
  else if (k == "res_wide") g_res_wide = (int)value;
  else if (k == "res_iss2") g_res_iss2 = (int)value;
  else if (k == "res_skew_iss2") g_res_skew_iss2 = (int)value;
  else if (k == "res_skew") g_res_skew = (int)value;
  else if (k == "res_ng") g_res_ng = (int)value;
  else if (k == "res_tb") g_res_tb = (int)value;
  else if (k == "res_gmax") g_res_gmax = (int)value;
  else if (k == "res_skew_pct") g_res_skew_pct = (int)value;
  else if (k == "pack") g_pk_on = (int)value;
  else if (k == "pk_mode") g_pk_mode = (int)value;
  else if (k == "pk_cg2") g_pk_cg2 = (int)value;
  else if (k == "pk_single_pct") g_pk_single_pct = (int)value;
  else if (k == "pk_fuse") g_pk_fuse_br = (int)value;
  else if (k == "pk_chan") g_pk_chan_mask = (int)value;
  else if (k == "cluster") g_knobs.cluster = value;
  else if (k == "alias_at") g_knobs.alias_at = value;
  else if (k == "epi_tma") g_knobs.epi_tma = value;
  else if (k == "pdl") g_tc_pdl = (int)value;
  else if (k == "pair_pref") g_pair_pref = (int)value;
  else if (k == "cg2") g_pair_cg2 = (int)value;
  else if (k == "pair_smem") g_knobs.pair_smem = value;
  else if (k == "trace_launch") g_knobs.trace_launch = value;
  else if (k == "span_ptr") g_knobs.span_ptr = value;
  else if (k == "plan_report") g_knobs.plan_report = value;
  else if (k == "trace_ptr") g_knobs.trace_ptr = value;
  else if (k == "max_msub") g_knobs.max_msub = value;
  else if (k == "max_nt") g_knobs.max_nt = value;
  else if (k == "tc_cg2") g_knobs.tc_cg2 = value;
  else if (k == "epi_pf") g_knobs.epi_pf = value;
  else if (k == "slab_cap") g_knobs.slab_cap = value;
  else if (k == "max_ctas") g_knobs.max_ctas = value;
  else if (k == "embed_tap") g_knobs.embed_tap = value;
  else if (k == "front_fuse") g_knobs.front_fuse = value;
  else if (k == "post_rows") g_knobs.post_rows = value;
  else if (k == "narrow_par") g_knobs.narrow_par = value;
  else if (k == "chain") g_knobs.chain = value;
  else if (k == "layer_events") g_knobs.layer_events = value;
  else if (k == "branch_par") g_knobs.branch_par = value;
  else if (k == "par_share") g_knobs.par_share = value;
  else return L2S_ERR_INVALID;
  return L2S_OK;
}

}  // extern "C"
