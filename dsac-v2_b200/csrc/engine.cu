// libdsact.so — host side of the B200-native DSAC-T update engine (C ABI in include/dsact.h).
//
// Orchestrates one `DSAC_V2.local_update` (reference dsac_v2.py:102-105,150-347) as a fixed sequence of
// kernel launches on caller-owned flat fp32 buffers, optionally captured once into a CUDA graph and
// replayed.  No CPU fallback: every entry point needs a CUDA device.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "../../include/dsact.h"
#include "gemm_simt.cuh"
#include "kernels.cuh"
#include "tc_host.cuh"
#include "chain_tc.cuh"
#include "dp_peer.cuh"
#include "replay_u8.cuh"

using namespace dsact;

static thread_local char g_err[512] = "";
static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
#define CUDA_TRY(x)                                                                       \
  do {                                                                                    \
    cudaError_t e_ = (x);                                                                 \
    if (e_ != cudaSuccess) return fail(DSACT_ECUDA, "%s failed: %s", #x, cudaGetErrorString(e_)); \
  } while (0)

// ---- network geometry -------------------------------------------------------
struct Net {
  int L;                                   // hidden layers
  int s[DSACT_MAX_HIDDEN + 2];             // s[0] input, s[1..L] hidden, s[L+1] output
  int64_t w[DSACT_MAX_HIDDEN + 1], b[DSACT_MAX_HIDDEN + 1], n;  // offsets inside the net, total floats
  void build(int in, const int32_t* hidden, int L_, int out) {
    L = L_;
    s[0] = in;
    for (int j = 0; j < L; ++j) s[j + 1] = hidden[j];
    s[L + 1] = out;
    n = 0;
    for (int j = 0; j <= L; ++j) {
      w[j] = n; n += (int64_t)s[j + 1] * s[j];
      b[j] = n; n += s[j + 1];
    }
  }
};

static int64_t round64(int64_t x) { return (x + 63) / 64 * 64; }

// bf16 image slot inside the arena (TC modes only)
struct ImgSlot {
  int64_t off = -1;  // floats from the workspace base
  int rows = 0, width = 0, pitch = 0;
  int64_t plane = 0;
};

// activation arena, all offsets in floats from the workspace base
struct Arena {
  int64_t obs, obs2, act, rew, done, logp, idx;    // gathered minibatch + int64 indices
  int64_t eps1, eps2, z3, z4;                      // device-generated noise
  int64_t zP[DSACT_MAX_HIDDEN], hP[DSACT_MAX_HIDDEN], hT[DSACT_MAX_HIDDEN], logitsP, logitsT;
  int64_t new_act, act2, logp_new, logp2;
  int64_t zQ[6][DSACT_MAX_HIDDEN], hQ[6][DSACT_MAX_HIDDEN], outQ[6];
  int64_t dOut[6], dzQ[6][DSACT_MAX_HIDDEN], dAct[2], dlogits, dzP[DSACT_MAX_HIDDEN];
  // ---- tcgen05 modes: bf16 hi/lo images of every GEMM operand + wgrad split slabs
  bool tc;
  ImgSlot i_obs, i_obs2, i_act, i_new_act, i_act2, i_dlogits;
  ImgSlot i_hP[DSACT_MAX_HIDDEN], i_hT[DSACT_MAX_HIDDEN], i_dzP[DSACT_MAX_HIDDEN];
  ImgSlot i_hQ[6][DSACT_MAX_HIDDEN], i_dzQ[6][DSACT_MAX_HIDDEN], i_dOut[6];
  ImgSlot i_wq[4][DSACT_MAX_HIDDEN + 1], i_wpi[2][DSACT_MAX_HIDDEN + 1];  // q1,q2,q1',q2' / pi,pi'
  int kpad_q0;        // column of the act block inside the Q layer-0 weight image
  int64_t slabs;      // [nslabs][n_params] fp32 wgrad partials
  int nslabs;
  int64_t slab_stride;   // floats between slabs: n_params rounded up to 4 (float4 access to every slab)
  int64_t total;
  void build(const dsact_config& c, const Net& q, const Net& pi) {
    int64_t B = c.max_batch, O = c.obs_dim, A = c.act_dim, off = 0;
    auto take = [&](int64_t n) { int64_t o = off; off += round64(n); return o; };
    auto img = [&](int rows, int width) {
      ImgSlot s;
      s.rows = rows; s.width = width; s.pitch = (width + 7) / 8 * 8;
      s.plane = round64((int64_t)rows * s.pitch);  // elements per plane, multiple of 64
      s.off = take(s.plane);  // 2 planes of bf16 = plane floats
      return s;
    };
    obs = take(B * O); obs2 = take(B * O); act = take(B * A); rew = take(B); done = take(B); logp = take(B); idx = take(2 * B);
    eps1 = take(B * A); eps2 = take(B * A); z3 = take(B); z4 = take(B);
    for (int j = 0; j < pi.L; ++j) { zP[j] = take(B * pi.s[j + 1]); hP[j] = take(B * pi.s[j + 1]); hT[j] = take(B * pi.s[j + 1]); dzP[j] = take(B * pi.s[j + 1]); }
    logitsP = take(B * 2 * A); logitsT = take(B * 2 * A); dlogits = take(B * 2 * A);
    new_act = take(B * A); act2 = take(B * A); logp_new = take(B); logp2 = take(B);
    for (int p = 0; p < 6; ++p) {
      for (int j = 0; j < q.L; ++j) { zQ[p][j] = take(B * q.s[j + 1]); hQ[p][j] = take(B * q.s[j + 1]); dzQ[p][j] = take(B * q.s[j + 1]); }
      outQ[p] = take(B * 2); dOut[p] = take(B * 2);
    }
    dAct[0] = take(B * A); dAct[1] = take(B * A);
    tc = c.gemm_mode != DSACT_GEMM_FP32;
    nslabs = 0; slabs = 0; slab_stride = 0; kpad_q0 = (int)((O + 63) / 64 * 64);
    if (tc) {
      const int Bi = (int)B;
      i_obs = img(Bi, (int)O); i_obs2 = img(Bi, (int)O); i_act = img(Bi, (int)A); i_new_act = img(Bi, (int)A); i_act2 = img(Bi, (int)A);
      i_dlogits = img(Bi, 2 * (int)A);
      for (int j = 0; j < pi.L; ++j) { i_hP[j] = img(Bi, pi.s[j + 1]); i_hT[j] = img(Bi, pi.s[j + 1]); i_dzP[j] = img(Bi, pi.s[j + 1]); }
      for (int p = 0; p < 6; ++p) {
        for (int j = 0; j < q.L; ++j) { i_hQ[p][j] = img(Bi, q.s[j + 1]); i_dzQ[p][j] = img(Bi, q.s[j + 1]); }
        i_dOut[p] = img(Bi, 2);
      }
      for (int n = 0; n < 4; ++n)
        for (int j = 0; j <= q.L; ++j) i_wq[n][j] = img(q.s[j + 1], j == 0 ? kpad_q0 + (int)A : q.s[j]);
      for (int n = 0; n < 2; ++n)
        for (int j = 0; j <= pi.L; ++j) i_wpi[n][j] = img(pi.s[j + 1], pi.s[j]);
      // batch split of the weight-gradient GEMMs: at most 4 slabs of >= 256 rows (about one wave of CTAs at B = 4096;
      // 8 slabs of 512 rows measured 5 % slower end to end: twice the partial tiles to write and to fold in apply)
      nslabs = (int)(B / 256); if (nslabs > 4) nslabs = 4; if (nslabs < 1) nslabs = 1;
      if (getenv("DSACT_WG_SLABS")) { const int v = atoi(getenv("DSACT_WG_SLABS")); if (v >= 1 && v <= 16 && v * 128 <= B) nslabs = v; }   // tuning aid
      slab_stride = (2 * q.n + pi.n + 1 + 3) / 4 * 4;
      slabs = take((int64_t)nslabs * slab_stride);
    }
    total = off;
  }
};

struct GraphKey {
  int kind; const void* p[9]; int32_t batch; int64_t gb; int64_t size; const void* idx;
  bool operator==(const GraphKey& o) const { return memcmp(this, &o, sizeof(GraphKey)) == 0; }
};
struct GraphEntry { GraphKey key; cudaGraphExec_t exec; int launches; uint64_t stamp; };

struct dsact_handle {
  dsact_config cfg;
  int device, num_sms;
  Net q, pi;
  Arena ar;
  dsact_buffers buf;
  dsact_replay rb;
  bool bound, rb_bound;
  uint64_t seed;
  int64_t dev_iter;          // what state[ST_ITER] will hold when the next enqueued work runs (-1 unknown)
  int32_t pending_batch;     // rows of the shard phase1 processed (phase2 must match)
  dsact_batch pending;       // batch pointers of phase1
  const float *pending_eps1, *pending_z3, *pending_z4;  // noise phase1 used (phase2 needs it again)
  int64_t dev_rb_size;       // what state[ST_RB_SIZE] holds
  bool join_pending = false; // a forked branch of the current enqueue has not been joined yet
  bool apply_early = false;  // phase 2 of the current enqueue already ran the critics' part of the update
  bool arena_imaged;         // the last dsact_replay_sample left bf16 images of obs/obs2/act beside the arena batch
  cudaStream_t cap_stream;   // capture-only stream
  cudaStream_t side_stream;  // second branch inside a step (critic weight gradients || policy backward chain)
  cudaEvent_t ev_fork, ev_join;
  cudaEvent_t ev_pro_fork, ev_pro_join;   // prologue branch (weight images, noise, clears) beside the replay gather
  cudaEvent_t ev_dp_fork, ev_dp_join;     // std-sum exchange of the data-parallel step beside the second forward chain
  // peer-memory data parallelism (dp_peer.cuh)
  float* dp_buf = nullptr;            // this rank's exchange buffer (cudaMalloc, exported with CUDA IPC)
  void* dp_opened[DP_MAX_RANKS] = {}; // peers' buffers as opened here
  DpComm dp = {};
  bool dp_ready = false;
  // host-minibatch staging (dsact_stage_host): two device sets + a private copy stream
  float* stage_buf[2] = {nullptr, nullptr};
  int64_t stage_floats = 0;
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_stage_ready[2] = {nullptr, nullptr}, ev_stage_done[2] = {nullptr, nullptr};
  bool stage_done_valid[2] = {false, false};
  int stage_turn = 0, stage_held = -1;
  bool tc_attr_done = false, chain_attr_done = false;   // cudaFuncSetAttribute is per device: tracked per handle
  TcGroup tc_scratch;                                   // host-side lowering scratch of launch_tc (~5 KiB)
  std::vector<GraphEntry> graphs;
  uint64_t stamp;
  int64_t launches;
  int32_t last_launches;
  bool tc() const { return cfg.gemm_mode != DSACT_GEMM_FP32; }
  bool fused() const {  // layer-chain kernel: every layer must fit one 256-column TMEM accumulator / A operand
    if (!tc() || getenv("DSACT_NO_FUSE")) return false;
    for (int j = 1; j <= q.L + 1; ++j) if (q.s[j] > 256) return false;
    for (int j = 1; j <= pi.L + 1; ++j) if (pi.s[j] > 256) return false;
    for (int j = 1; j <= q.L; ++j) if (q.s[j] % 8) return false;    // hidden widths: 16-byte strides for the TMA epilogue
    for (int j = 1; j <= pi.L; ++j) if (pi.s[j] % 8) return false;
    return cfg.act_dim <= 256;
  }
  int passes() const { return cfg.gemm_mode == DSACT_GEMM_BF16X3 ? 3 : 1; }
  float* W() const { return reinterpret_cast<float*>(buf.workspace); }
  Img img(const ImgSlot& s, int rows) const {  // image handle with the live row count
    Img i;
    if (s.off < 0) return i;
    i.p = reinterpret_cast<__nv_bfloat16*>(W() + s.off);
    i.rows = rows; i.width = s.width; i.pitch = s.pitch; i.plane = s.plane;
    return i;
  }
};

enum { CLS_OTHER = 0, CLS_GEMM_FWD = 1, CLS_GEMM_DGRAD = 2, CLS_GEMM_WGRAD = 3, CLS_COUNT = 4 };
struct Prof {  // dsact_profile_step: an event after every launch
  std::vector<cudaEvent_t> ev;
  std::vector<int> cls;
  std::vector<double> flops;
};
struct Ctx {
  cudaStream_t s;
  int launches;
  cudaError_t err;
  Prof* prof = nullptr;
  cudaStream_t side = nullptr;   // optional second stream for an independent branch (null: serialise on `s`)
  bool pdl = true;               // programmatic dependent launch for this enqueue (off in fp32 mode, see pdl_enabled)
  void check() { cudaError_t e = cudaGetLastError(); if (e != cudaSuccess && err == cudaSuccess) err = e; }
  void done(int cls = CLS_OTHER, double flops = 0.0) {
    launches++;
    if (prof) {
      cudaEvent_t e;
      cudaEventCreate(&e);
      cudaEventRecord(e, s);
      prof->ev.push_back(e);
      prof->cls.push_back(cls);
      prof->flops.push_back(flops);
    }
  }
};

// Every kernel goes out with the programmatic-dependent-launch attribute (each kernel begins with griddepcontrol.wait),
// so that inside the captured graph a kernel's launch and prologue overlap its predecessor's tail (measured: -18 us of
// a 280 us step at B=4096, tools/pdl_ab.sh).  DSACT_PDL=0 turns it off.  The fp32 SIMT mode launches without it: its
// multi-wave GEMM grids lose SM slots to early-launched dependents (measured 514 vs 566 steps/s).
static bool pdl_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("DSACT_PDL"); v = (e && e[0] == '0') ? 0 : 1; }
  return v == 1;
}
template <typename... KArgs, typename... Args>
static void launch_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, Ctx& c, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = c.s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = (pdl_enabled() && c.pdl) ? 1 : 0;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
  if (e != cudaSuccess && c.err == cudaSuccess) c.err = e;
}

// ---- GEMM group launch -------------------------------------------------------
enum { V_FWD = 0, V_DGRAD = 1, V_WGRAD = 2 };

// A group of independent problems in both lowerings: fp32 pointers (GemmGroup) and bf16 images (TcExtra).
struct Group {
  GemmGroup g;               // SIMT lowering holds at most MAXG problems per launch; tcgen05 up to TC_MAXG
  GemmProb more[TC_MAXG - MAXG];
  TcExtra x[TC_MAXG];
  int n = 0;
  GemmProb& prob(int i) { return i < MAXG ? g.p[i] : more[i - MAXG]; }
  const GemmProb& prob(int i) const { return i < MAXG ? g.p[i] : more[i - MAXG]; }
  float* wg_slab = nullptr;   // wgrad split slabs (default: the arena's, addressed like the gradient buffer)
  long long wg_stride = 0;
  int wg_nslabs = 0;
  Group() { g.n = 0; }
  void push(const GemmProb& p, const TcExtra& e) { x[n] = e; prob(n) = p; ++n; g.n = n < MAXG ? n : MAXG; }
};

template <int BM, int BN>
static void launch_variant(const GemmGroup& g, int variant, int grid, Ctx& c) {
  if (variant == V_FWD) launch_k(gemm_kernel<BM, BN, true, true>, grid, 256, 0, c, g);
  else if (variant == V_DGRAD) launch_k(gemm_kernel<BM, BN, true, false>, grid, 256, 0, c, g);
  else launch_k(gemm_kernel<BM, BN, false, false>, grid, 256, 0, c, g);
}

static void launch_simt(int num_sms, GemmGroup& g, int variant, Ctx& c) {
  auto count = [&](int T) {
    int total = 0;
    for (int i = 0; i < g.n; ++i) total += ((g.p[i].M + T - 1) / T) * ((g.p[i].N + T - 1) / T);
    return total;
  };
  const bool big = variant != V_WGRAD && count(128) >= num_sms;
  const int T = big ? 128 : 64;
  const int base = count(T);
  int grid = 0;
  for (int i = 0; i < g.n; ++i) {
    GemmProb& p = g.p[i];
    p.tiles_m = (p.M + T - 1) / T;
    p.tiles_n = (p.N + T - 1) / T;
    p.ksplit = 1;
    if (variant == V_WGRAD) {  // reduction over the batch: split it until ~2 CTAs per SM, >= 4 k-tiles each
      const int nt = (p.K[0] + KT - 1) / KT;
      int want = (2 * num_sms + base - 1) / base;
      int maxs = nt / 4 > 0 ? nt / 4 : 1;
      p.ksplit = want < maxs ? want : maxs;
      if (p.ksplit < 1) p.ksplit = 1;
      const int per = (nt + p.ksplit - 1) / p.ksplit;
      p.ksplit = (nt + per - 1) / per;  // no empty splits
    }
    p.tile_start = grid;
    grid += p.tiles_m * p.tiles_n * p.ksplit;
  }
  if (big) launch_variant<128, 128>(g, variant, grid, c);
  else launch_variant<64, 64>(g, variant, grid, c);
}

// Lower the group onto tcgen05: images instead of fp32 operands, TMA tensor maps, 128 x bn tiles.
// `max_ctas` > 0: issue the group as several launches of at most that many CTAs (one CTA occupies an SM), which leaves
// the remaining SMs to a concurrent branch of the step graph for the whole duration.
static void launch_tc(dsact_handle* h, Group& G, int variant, Ctx& c, int max_ctas = 0) {
  TcGroup& t = h->tc_scratch;
  memset(&t, 0, sizeof(t));
  t.n = G.n;
  t.passes = h->passes();
  const bool a_mn = variant == V_WGRAD, b_mn = variant != V_FWD;
  int grid = 0;
  int bn_max = 16;
  int wg_bn = 128;
  if (variant == V_WGRAD) {  // a launch that would leave most SMs idle at 128-wide tiles gets 64-wide ones
    int ctas = 0;
    for (int i = 0; i < G.n; ++i) ctas += ((G.prob(i).M + TC_BM - 1) / TC_BM) * ((G.prob(i).N + 127) / 128) * (G.wg_slab ? G.wg_nslabs : h->ar.nslabs);
    if (ctas * 2 <= h->num_sms) wg_bn = 64;
    if (getenv("DSACT_WG_BN")) { const int v = atoi(getenv("DSACT_WG_BN")); if (v == 64 || v == 128 || v == 256) wg_bn = v; }   // tuning aid
  }
  for (int i = 0; i < G.n; ++i) {
    const GemmProb& s = G.prob(i);
    const TcExtra& x = G.x[i];
    TcProb& p = t.p[i];
    p.M = s.M; p.N = s.N;
    int bn = (s.N + 15) / 16 * 16;
    if (bn > 256) bn = 256;
    if (variant == V_WGRAD && bn > wg_bn) bn = wg_bn;  // more tiles for the (few, batch-split) weight-gradient problems
    p.bn = bn;
    if (bn > bn_max) bn_max = bn;
    p.tiles_m = (s.M + TC_BM - 1) / TC_BM;
    p.tiles_n = (s.N + bn - 1) / bn;
    for (int sgm = 0; sgm < 2; ++sgm) {
      p.kblocks[sgm] = (s.K[sgm] + TC_BK - 1) / TC_BK;
      p.kB0[sgm] = x.kB0[sgm];
      if (s.K[sgm] > 0 && !make_map(&p.mapA[sgm], x.a[sgm], a_mn ? 64 : TC_BM)) { c.err = cudaErrorInvalidValue; return; }
    }
    if (!make_map(&p.mapB, x.b, b_mn ? 64 : bn)) { c.err = cudaErrorInvalidValue; return; }
    p.ksplit = 1;
    p.C = s.C; p.ldc = s.ldc; p.bias = s.bias; p.Zout = s.Zout; p.Zin = s.Zin; p.ldz = s.ldz; p.colsum = s.colsum;
    p.epi = s.epi; p.act = s.act;
    if (variant == V_WGRAD) {  // fixed slab count: empty splits store zeros so that the reduction is always valid
      p.epi = EPI_PARTIAL;
      if (G.wg_slab) { p.ksplit = G.wg_nslabs; p.C = G.wg_slab; p.split_stride = G.wg_stride; }
      else {
        p.ksplit = h->ar.nslabs;
        p.C = h->W() + h->ar.slabs + (s.C - h->buf.grads);
        p.split_stride = h->ar.slab_stride;
      }
    }
    if (x.out.p) {
      p.img = x.out.p; p.img_pitch = x.out.pitch; p.img_plane = x.out.plane;
      if (p.epi == EPI_BIAS_ACT || p.epi == EPI_DACT) p.C = nullptr;  // the next GEMM reads the image; no fp32 copy
    }
    p.tile_start = grid;
    grid += p.tiles_m * p.tiles_n * p.ksplit;
  }
  static unsigned long long* dbg = nullptr;
  const bool debug = getenv("DSACT_TC_DEBUG") != nullptr;
  if (debug && !dbg) cudaMalloc(&dbg, sizeof(unsigned long long) * TC_DBG_SLOTS * 4096);
  if (debug && grid <= 4096) { cudaMemsetAsync(dbg, 0, sizeof(unsigned long long) * TC_DBG_SLOTS * grid, c.s); t.dbg = dbg; }
  const int planes = t.passes == 3 ? 2 : 1;
  const int stage_b = (b_mn ? (bn_max + 63) / 64 * 64 : bn_max) * 128;   // bytes of one B plane per stage
  int stages = (200 * 1024) / (planes * (TC_STAGE_A + stage_b));
  if (stages > 8) stages = 8;
  const int smem = tc_smem_bytes(stages, planes, stage_b);
  if (!h->tc_attr_done) {
    cudaFuncSetAttribute(tc_gemm_kernel<false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    cudaFuncSetAttribute(tc_gemm_kernel<false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    cudaFuncSetAttribute(tc_gemm_kernel<true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    cudaFuncSetAttribute(tc_gemm_kernel<false, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    cudaFuncSetAttribute(tc_gemm_kernel<false, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    cudaFuncSetAttribute(tc_gemm_kernel<true, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    h->tc_attr_done = true;
  }
  const int total = grid;
  if (max_ctas > 0 && !debug && total > max_ctas) {  // equal slices, none above the bound
    const int parts = (total + max_ctas - 1) / max_ctas;
    grid = (total + parts - 1) / parts;
  }
  for (int t0 = 0; t0 < total; t0 += grid) {
    t.tile0 = t0;
    const int n = total - t0 < grid ? total - t0 : grid;
    if (t0 > 0) c.launches++;
    if (planes == 2) {
      if (variant == V_FWD) launch_k(tc_gemm_kernel<false, false, true>, n, TC_THREADS, smem, c, t, stages, stage_b);
      else if (variant == V_DGRAD) launch_k(tc_gemm_kernel<false, true, true>, n, TC_THREADS, smem, c, t, stages, stage_b);
      else launch_k(tc_gemm_kernel<true, true, true>, n, TC_THREADS, smem, c, t, stages, stage_b);
    } else {
      if (variant == V_FWD) launch_k(tc_gemm_kernel<false, false, false>, n, TC_THREADS, smem, c, t, stages, stage_b);
      else if (variant == V_DGRAD) launch_k(tc_gemm_kernel<false, true, false>, n, TC_THREADS, smem, c, t, stages, stage_b);
      else launch_k(tc_gemm_kernel<true, true, false>, n, TC_THREADS, smem, c, t, stages, stage_b);
    }
  }
  grid = total;
  if (debug && t.dbg) {  // per-CTA phase breakdown (ns): setup | first TMA landed | MMA issue done | accumulator ready | epilogue | teardown
    cudaStreamSynchronize(c.s);
    std::vector<unsigned long long> hbuf(TC_DBG_SLOTS * (size_t)grid);
    cudaMemcpy(hbuf.data(), dbg, sizeof(unsigned long long) * TC_DBG_SLOTS * grid, cudaMemcpyDeviceToHost);
    unsigned long long tmin = ~0ull, tmax = 0;
    double ph[6] = {0, 0, 0, 0, 0, 0};
    for (int i = 0; i < grid; ++i) {
      const unsigned long long* d = &hbuf[TC_DBG_SLOTS * (size_t)i];
      if (d[0] < tmin) tmin = d[0];
      if (d[6] > tmax) tmax = d[6];
      ph[0] += (double)(d[1] - d[0]); ph[1] += (double)(d[2] - d[1]); ph[2] += (double)(d[3] - d[2]);
      ph[3] += (double)(d[4] - d[3]); ph[4] += (double)(d[5] - d[4]); ph[5] += (double)(d[6] - d[5]);
    }
    fprintf(stderr, "[tc_debug] variant %d grid %d span %.1f us | per-CTA avg ns: setup %.0f, first-load %.0f, mma-issue %.0f, acc-wait %.0f, epilogue %.0f, teardown %.0f\n",
            variant, grid, (tmax - tmin) / 1000.0, ph[0] / grid, ph[1] / grid, ph[2] / grid, ph[3] / grid, ph[4] / grid, ph[5] / grid);
  }
}

static void launch_group(dsact_handle* h, Group& G, int variant, Ctx& c, int max_ctas = 0) {
  if (G.n == 0) return;
  double flops = 0.0;
  for (int i = 0; i < G.n; ++i) flops += 2.0 * G.prob(i).M * G.prob(i).N * ((double)G.prob(i).K[0] + G.prob(i).K[1]);
  if (h->tc()) {
    launch_tc(h, G, variant, c, max_ctas);
    c.done(CLS_GEMM_FWD + variant, flops);
  } else {
    G.g.n = G.n < MAXG ? G.n : MAXG;
    launch_simt(h->num_sms, G.g, variant, c);
    c.done(CLS_GEMM_FWD + variant, flops);
    if (G.n > MAXG) {  // second launch for the overflow
      GemmGroup g2;
      g2.n = G.n - MAXG;
      for (int i = 0; i < g2.n; ++i) g2.p[i] = G.more[i];
      launch_simt(h->num_sms, g2, variant, c);
      c.done(CLS_GEMM_FWD + variant, 0.0);
    }
  }
  c.check();
}

static GemmProb prob_zero() {
  GemmProb p;
  memset(&p, 0, sizeof(p));
  return p;
}

// a [rows, ld] tensor as both lowerings see it
struct Ten {
  float* f = nullptr;
  Img im;
};
struct Wt {       // one layer's weights: fp32 [out, in] + image
  const float* f = nullptr;
  const float* bias = nullptr;
  Img im;
};

// forward layer j: out = act(in0 * W[:, :k0]^T + in1 * W[:, k0:k0+k1]^T + b)
static void add_fwd(Group& G, const Net& net, int j, const Wt& w, const Ten& in0, int k0, const Ten& in1, int k1, int kB1,
                    const Ten& out, float* zout, int B, int act) {
  GemmProb p = prob_zero();
  TcExtra x;
  const int in_dim = net.s[j];
  p.A[0] = in0.f; p.lda[0] = k0; p.K[0] = k0; p.B[0] = w.f; p.ldb[0] = in_dim;
  x.a[0] = in0.im;
  if (k1 > 0) {
    p.A[1] = in1.f; p.lda[1] = k1; p.K[1] = k1; p.B[1] = w.f + k0; p.ldb[1] = in_dim;
    x.a[1] = in1.im; x.kB0[1] = kB1;
  }
  x.b = w.im;
  p.M = B; p.N = net.s[j + 1]; p.C = out.f; p.ldc = net.s[j + 1];
  p.bias = w.bias;
  const bool last = j == net.L;
  p.epi = last ? EPI_STORE : EPI_BIAS_ACT;
  p.act = act;
  p.Zout = last ? nullptr : zout;
  x.out = last ? Img() : out.im;
  G.push(p, x);
}

// dgrad through layer j, weight columns [col0, col0+ncols): dX = dY * W[:, cols]   (* act'(Zprev), bias-grad colsum)
static void add_dgrad(Group& G, const Net& net, int j, const Wt& w, int col0, int img_col0, int ncols, const Ten& dY,
                      const Ten& dX, const float* Zprev, float* gbias_prev, int B, int act) {
  GemmProb p = prob_zero();
  TcExtra x;
  p.A[0] = dY.f; p.lda[0] = net.s[j + 1]; p.K[0] = net.s[j + 1];
  p.B[0] = w.f + col0; p.ldb[0] = net.s[j];
  x.a[0] = dY.im;
  x.b = w.im.cols(img_col0, ncols);
  p.M = B; p.N = ncols; p.C = dX.f; p.ldc = ncols;
  if (Zprev) { p.epi = EPI_DACT; p.Zin = Zprev; p.ldz = ncols; p.colsum = gbias_prev; p.act = act; }
  else p.epi = EPI_STORE;
  x.out = dX.im;
  G.push(p, x);
}

// wgrad of layer j, weight columns [col0, col0+ncols): gW[:, cols] += dY^T X
static void add_wgrad(Group& G, const Net& net, int j, float* Gw, int col0, int ncols, const Ten& dY, const Ten& X, int B) {
  GemmProb p = prob_zero();
  TcExtra x;
  p.A[0] = dY.f; p.lda[0] = net.s[j + 1]; p.K[0] = B;
  p.B[0] = X.f; p.ldb[0] = ncols;
  x.a[0] = dY.im; x.b = X.im;
  p.M = net.s[j + 1]; p.N = ncols; p.C = Gw + col0; p.ldc = net.s[j];
  p.epi = EPI_ATOMIC;
  G.push(p, x);
}

// fp32 -> image conversions (TC modes)
struct ImgBatch {
  ImgGroup g;
  bool overflow = false;
  ImgBatch() { g.n = 0; }
  void add(const float* src, int ld_src, const Img& dst, int rows, int w0, int w1 = 0, int dst1 = 0) {
    if (g.n >= IMG_MAXJ) { overflow = true; return; }
    ImgJob& j = g.j[g.n++];
    memset(&j, 0, sizeof(j));
    j.src = src; j.dst = dst.p; j.rows = rows; j.ld_src = ld_src;
    j.seg_w[0] = w0; j.seg_src0[0] = 0; j.seg_dst0[0] = 0;
    j.seg_w[1] = w1; j.seg_src0[1] = w0; j.seg_dst0[1] = dst1;
    j.pitch = dst.pitch; j.fill_w = w1 > 0 ? dst1 + w1 : w0; j.plane = dst.plane;
  }
  void reserve(const dsact_handle* h, Ctx& c, int jobs) { if (g.n + jobs > IMG_MAXJ) launch(h, c); }   // flush when full
  // `pro` != null: the clears and the device noise ride in the same launch (step_prologue_kernel)
  void launch(const dsact_handle* h, Ctx& c, PrologueArgs* pro = nullptr) {
    if (overflow) { c.err = cudaErrorInvalidValue; return; }
    if (g.n == 0 && !pro) return;
    g.planes = h->passes() == 3 ? 2 : 1;
    int grid = 0;
    for (int i = 0; i < g.n; ++i) {
      g.j[i].block_start = grid;
      long long total = (long long)g.j[i].rows * (g.j[i].pitch / 8);
      int blocks = (int)((total + 255) / 256);
      if (blocks < 1) blocks = 1;
      if (blocks > 2 * h->num_sms) blocks = 2 * h->num_sms;
      grid += blocks;
    }
    if (pro) {
      pro->img_blocks = grid;
      launch_k(step_prologue_kernel, grid + pro->zero_blocks + pro->noise_blocks, 256, 0, c, g, *pro);
    } else {
      launch_k(image_kernel, grid, 256, 0, c, g);
    }
    c.done();
    g.n = 0;
  }
};

static ImgOut img_out(const dsact_handle* h, const ImgSlot& s) {
  ImgOut o;
  o.p = nullptr; o.pitch = 0; o.planes = h->passes() == 3 ? 2 : 1; o.plane = 0;
  if (h->tc() && s.off >= 0) { o.p = reinterpret_cast<__nv_bfloat16*>(h->W() + s.off); o.pitch = s.pitch; o.plane = s.plane; }
  return o;
}

static Wt weight(const dsact_handle* h, const Net& net, const float* base, int j, const ImgSlot& slot) {
  Wt w;
  w.f = base + net.w[j];
  w.bias = base + net.b[j];
  w.im = h->img(slot, net.s[j + 1]);
  return w;
}


// ---- layer-chain launches (tcgen05 modes) -------------------------------------------------------
struct ChainBuild {
  ChainGroup g;
  int grid = 0, stage_b = 16 * 128;
  double flops = 0.0;
  bool ok = true;
  explicit ChainBuild(int passes) { memset(&g, 0, sizeof(g)); g.passes = passes; }
  ChainPass& begin(const Img& a0, const Img& a1, int M) {
    ChainPass& P = g.p[g.n++];
    P.n_layers = 0; P.M = M; P.tile_start = grid;
    grid += (M + TC_BM - 1) / TC_BM;
    ok = ok && make_map(&P.mapA[0], a0, TC_BM);
    if (a1.p) ok = ok && make_map(&P.mapA[1], a1, TC_BM);
    return P;
  }
  ChainLayer& layer(ChainPass& P, const Img& wimg, bool b_mn, int N, int K0, int K1, int kB1) {
    ChainLayer& L = P.L[P.n_layers++];
    L.N = N; L.bn = (N + 15) / 16 * 16; L.b_mn = b_mn ? 1 : 0;
    L.kblocks[0] = (K0 + TC_BK - 1) / TC_BK; L.kblocks[1] = (K1 + TC_BK - 1) / TC_BK;
    L.kB0[0] = 0; L.kB0[1] = kB1; L.K = K0;
    ok = ok && make_map(&L.mapB, wimg, b_mn ? 64 : L.bn);
    const int sb = b_mn ? (L.bn + 63) / 64 * 8192 : L.bn * 128;
    if (sb > stage_b) stage_b = sb;
    flops += 2.0 * P.M * N * ((double)K0 + K1);
    return L;
  }
};

static void launch_chain(dsact_handle* h, ChainBuild& cb, int cls, Ctx& c) {
  if (cb.g.n == 0) return;
  if (!cb.ok) { c.err = cudaErrorInvalidValue; return; }
  static unsigned long long* dbg = nullptr;
  const bool debug = getenv("DSACT_TC_DEBUG") != nullptr;
  if (debug && !dbg) cudaMalloc(&dbg, sizeof(unsigned long long) * TC_DBG_SLOTS * 4096);
  if (debug && cb.grid <= 4096) { cudaMemsetAsync(dbg, 0, sizeof(unsigned long long) * TC_DBG_SLOTS * cb.grid, c.s); cb.g.dbg = dbg; }
  const int planes = cb.g.passes == 3 ? 2 : 1;
  const int stages = planes == 2 ? 2 : 3;
  const int smem = chain_smem_bytes(stages, planes, cb.stage_b);
  if (!h->chain_attr_done) {
    cudaFuncSetAttribute(tc_chain_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    cudaFuncSetAttribute(tc_chain_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    h->chain_attr_done = true;
  }
  if (planes == 2) launch_k(tc_chain_kernel<true>, cb.grid, TC_THREADS, smem, c, cb.g, stages, cb.stage_b);
  else launch_k(tc_chain_kernel<false>, cb.grid, TC_THREADS, smem, c, cb.g, stages, cb.stage_b);
  c.done(cls, cb.flops);
  c.check();
  if (debug && cb.g.dbg) {
    cudaStreamSynchronize(c.s);
    std::vector<unsigned long long> hbuf(TC_DBG_SLOTS * (size_t)cb.grid);
    cudaMemcpy(hbuf.data(), dbg, sizeof(unsigned long long) * TC_DBG_SLOTS * cb.grid, cudaMemcpyDeviceToHost);
    unsigned long long tmin = ~0ull, tmax = 0;
    for (int i = 0; i < cb.grid; ++i) {
      const unsigned long long* d = &hbuf[TC_DBG_SLOTS * (size_t)i];
      if (d[0] < tmin) tmin = d[0];
      if (d[6] > tmax) tmax = d[6];
    }
    fprintf(stderr, "[chain_debug] class %d passes %d grid %d span %.1f us\n", cls, cb.g.n, cb.grid, (tmax - tmin) / 1000.0);
    for (int pi = 0; pi < cb.g.n; ++pi) {  // first CTA of every pass: per-layer timeline relative to its start (us)
      const unsigned long long* d = &hbuf[TC_DBG_SLOTS * (size_t)cb.g.p[pi].tile_start];
      fprintf(stderr, "  pass %d: setup %.1f first-load %.1f |", pi, (d[1] - d[0]) / 1e3, (d[2] - d[0]) / 1e3);
      for (int j = 0; j < cb.g.p[pi].n_layers; ++j)
        fprintf(stderr, " L%d mma-issued %.1f acc-ready %.1f epi-done %.1f |", j, (d[8 + 3 * j] - d[0]) / 1e3, (d[9 + 3 * j] - d[0]) / 1e3,
                (d[10 + 3 * j] - d[0]) / 1e3);
      fprintf(stderr, " end %.1f\n", (d[6] - d[0]) / 1e3);
      if (d[32] && d[38])   // first chunk of layer 1, first epilogue warp (SM cycles): ld | math | split | stage+TMA | st+arrive ; whole layer
        fprintf(stderr, "    L1 chunk0 cycles: ld %lld math %lld split %lld stage %lld st+arrive %lld | layer (4 chunks) %lld\n",
                (long long)(d[33] - d[32]), (long long)(d[34] - d[33]), (long long)(d[35] - d[34]), (long long)(d[36] - d[35]),
                (long long)(d[37] - d[36]), (long long)(d[38] - d[32]));
      if (d[39] && d[41])   // inside "stage": wait for the previous stores' reads | STS | proxy fence | TMA store issue
        fprintf(stderr, "    L1 chunk0 stage cycles: wait_read %lld sts %lld fence %lld tma-issue %lld\n", (long long)(d[39] - d[35]),
                (long long)(d[40] - d[39]), (long long)(d[41] - d[40]), (long long)(d[36] - d[41]));
    }
  }
}

// forward chain of one pass: out = head(act(...act(in W_0^T + b_0)...))
static ChainPass& chain_fwd_pass(ChainBuild& cb, const dsact_handle* h, const Net& net, const float* Wbase, const ImgSlot* wslots,
                           const Img& in0, int k0, const Img& in1, int k1, int kB1, int B, int act,
                           const int64_t* zout_off, const ImgSlot* himg, float* out) {
  ChainPass& P = cb.begin(in0, in1, B);
  float* W = h->W();
  for (int j = 0; j <= net.L; ++j) {
    const Img wim = h->img(wslots[j], net.s[j + 1]);
    ChainLayer& L = j == 0 ? cb.layer(P, wim, false, net.s[1], k0, k1, kB1) : cb.layer(P, wim, false, net.s[j + 1], net.s[j], 0, 0);
    const bool last = j == net.L;
    L.epi = last ? EPI_STORE : EPI_BIAS_ACT;
    L.act = act;
    L.bias = Wbase + net.b[j];
    if (last) L.C = out;
    else {
      if (zout_off) { L.Zout = W + zout_off[j]; cb.ok = cb.ok && make_map_f32(&L.mapZ, L.Zout, B, net.s[j + 1], net.s[j + 1]); }
      if (himg) {
        const Img im = h->img(himg[j], B);
        L.img = im.p; L.img_pitch = im.pitch; L.img_plane = im.plane;
        cb.ok = cb.ok && make_map_img_store(&L.mapImg, im, h->passes() == 3 ? 2 : 1);
      }
    }
  }
  return P;
}

// dgrad chain of one pass: dz_{j-1} = (dz_j W_j) (.) act'(z_{j-1}) for j = L..1 (+ dAct = dz_0 W_0[:, act columns])
static ChainPass& chain_dgrad_pass(ChainBuild& cb, const dsact_handle* h, const Net& net, const ImgSlot* wslots, const Img& dout,
                             int B, int act, const int64_t* zin_off, float* gbase /*bias grads of this net or null*/,
                             const ImgSlot* dzimg /*or null*/, float* dact_out, int act_col_img, int act_cols) {
  const Img none;
  ChainPass& P = cb.begin(dout, none, B);
  float* W = h->W();
  for (int j = net.L; j >= 1; --j) {
    const Img wim = h->img(wslots[j], net.s[j + 1]);   // rows = reduction (outputs of layer j), width = inputs
    ChainLayer& L = cb.layer(P, wim, true, net.s[j], net.s[j + 1], 0, 0);
    L.epi = EPI_DACT; L.act = act;
    L.Zin = W + zin_off[j - 1];
    cb.ok = cb.ok && make_map_f32(&L.mapZ, L.Zin, B, net.s[j], net.s[j]);
    L.colsum = gbase ? gbase + net.b[j - 1] : nullptr;
    if (dzimg) {
      const Img im = h->img(dzimg[j - 1], B);
      L.img = im.p; L.img_pitch = im.pitch; L.img_plane = im.plane;
      cb.ok = cb.ok && make_map_img_store(&L.mapImg, im, h->passes() == 3 ? 2 : 1);
    }
  }
  if (dact_out) {
    const Img wim = h->img(wslots[0], net.s[1]).cols(act_col_img, act_cols);
    ChainLayer& L = cb.layer(P, wim, true, act_cols, net.s[1], 0, 0);
    L.epi = EPI_STORE; L.C = dact_out;
  }
  return P;
}

// ---- enqueue: pieces of one update ---------------------------------------------
// Everything of a step that depends on neither the minibatch gather nor a forward pass: accumulator clears, the
// gradient memset, the bf16 images of all weights (and of a caller-supplied batch), the device noise.
static void enqueue_noise(dsact_handle* h, int B, Ctx& c) {
  const Arena& ar = h->ar;
  float* W = h->W();
  const int A = h->cfg.act_dim;
  const int total = (B * A + 1) / 2 * 2 + (B + 1) / 2 * 2;
  int blocks = (total / 2 + 255) / 256; if (blocks < 1) blocks = 1;
  launch_k(noise_kernel, blocks, 256, 0, c, W + ar.eps1, W + ar.eps2, W + ar.z3, W + ar.z4, B, A, h->seed, h->buf.state);
  c.done();
}
static bool prologue_merged() {   // DSACT_PROLOGUE_MERGE=0: separate clear / image / noise launches (A/B aid)
  static const bool off = getenv("DSACT_PROLOGUE_MERGE") && getenv("DSACT_PROLOGUE_MERGE")[0] == '0';
  return !off;
}
static void enqueue_prologue(dsact_handle* h, const dsact_batch& bt, const dsact_noise* nz, Ctx& c, bool inputs_imaged,
                             bool with_noise = true) {
  const dsact_config& cf = h->cfg;
  const Net &q = h->q, &pi = h->pi;
  const Arena& ar = h->ar;
  float* W = h->W();
  const int B = bt.batch, O = cf.obs_dim, A = cf.act_dim;
  const bool tc = h->tc();
  float* P = h->buf.params;
  float* T = h->buf.targets;
  const float* Qb[4] = {P, P + q.n, T, T + q.n};        // q1, q2, q1', q2'
  const float* PIb[2] = {P + 2 * q.n, T + 2 * q.n};     // pi, pi'

  const long long n_grads = 2 * q.n + pi.n + 1;
  int zero_blocks = (int)((n_grads / 4 + 255) / 256); if (zero_blocks > 2 * h->num_sms) zero_blocks = 2 * h->num_sms; if (zero_blocks < 1) zero_blocks = 1;
  const bool want_noise = !nz && with_noise;
  const bool merged = tc && prologue_merged();   // tcgen05 modes: clears + images + noise as one launch
  if (!merged) { launch_k(begin_step_kernel, zero_blocks, 256, 0, c, h->buf.state, h->buf.grads, n_grads); c.done(); }

  if (tc) {  // refresh the weight images (the caller may have written params/targets through its views) + inputs
    ImgBatch ib;
    for (int n = 0; n < 2; ++n)
      for (int j = 0; j <= q.L; ++j) {
        ib.reserve(h, c, 1);
        const Img im = h->img(ar.i_wq[n][j], q.s[j + 1]);
        if (j == 0) ib.add(Qb[n] + q.w[0], O + A, im, q.s[1], O, A, ar.kpad_q0);
        else ib.add(Qb[n] + q.w[j], q.s[j], im, q.s[j + 1], q.s[j]);
      }
    ib.reserve(h, c, pi.L + 2);
    for (int j = 0; j <= pi.L; ++j) ib.add(PIb[0] + pi.w[j], pi.s[j], h->img(ar.i_wpi[0][j], pi.s[j + 1]), pi.s[j + 1], pi.s[j]);
    if (!inputs_imaged) ib.add(bt.obs, O, h->img(ar.i_obs, B), B, O);
    for (int n = 2; n < 4; ++n)
      for (int j = 0; j <= q.L; ++j) {
        ib.reserve(h, c, 1);
        const Img im = h->img(ar.i_wq[n][j], q.s[j + 1]);
        if (j == 0) ib.add(Qb[n] + q.w[0], O + A, im, q.s[1], O, A, ar.kpad_q0);
        else ib.add(Qb[n] + q.w[j], q.s[j], im, q.s[j + 1], q.s[j]);
      }
    ib.reserve(h, c, pi.L + 3);
    for (int j = 0; j <= pi.L; ++j) ib.add(PIb[1] + pi.w[j], pi.s[j], h->img(ar.i_wpi[1][j], pi.s[j + 1]), pi.s[j + 1], pi.s[j]);
    if (!inputs_imaged) {
      ib.add(bt.obs2, O, h->img(ar.i_obs2, B), B, O);
      ib.add(bt.act, A, h->img(ar.i_act, B), B, A);
    }
    if (merged) {
      PrologueArgs pa;
      memset(&pa, 0, sizeof(pa));
      pa.zero_blocks = zero_blocks;
      pa.state = h->buf.state; pa.grads = h->buf.grads; pa.n_grads = n_grads;
      pa.hy = AdamHyper{cf.lr_q, cf.lr_pi, cf.lr_alpha, cf.adam_beta1, cf.adam_beta2};
      if (want_noise) {
        const int total = (B * A + 1) / 2 * 2 + (B + 1) / 2 * 2;
        pa.noise_blocks = (total / 2 + 255) / 256; if (pa.noise_blocks < 1) pa.noise_blocks = 1;
        pa.eps1 = W + ar.eps1; pa.eps2 = W + ar.eps2; pa.z3 = W + ar.z3; pa.z4 = W + ar.z4;
        pa.B = B; pa.A = A; pa.seed = h->seed;
      }
      ib.launch(h, c, &pa);
    } else {
      ib.launch(h, c);
    }
  }

  // device noise; the counter it reads is stepped by sample_kernel, once every reader of this step has run
  if (want_noise && !merged) enqueue_noise(h, B, c);
  c.check();
}

// In a captured step the prologue runs as its own branch next to whatever the main stream does first (the replay
// gather); returns true if it was forked and must be joined (enqueue_phase1 does) before the first forward pass.
static bool fork_prologue(dsact_handle* h, const dsact_batch& bt, const dsact_noise* nz, Ctx& c, bool inputs_imaged) {
  if (!c.side) return false;
  cudaEventRecord(h->ev_pro_fork, c.s);
  cudaStreamWaitEvent(c.side, h->ev_pro_fork, 0);
  Ctx cs{c.side, 0, cudaSuccess};
  cs.pdl = c.pdl;
  enqueue_prologue(h, bt, nz, cs, inputs_imaged, true);
  cudaEventRecord(h->ev_pro_join, c.side);
  c.launches += cs.launches;
  if (cs.err != cudaSuccess && c.err == cudaSuccess) c.err = cs.err;
  return true;
}

static unsigned long long dp_timeout_ns() {
  static const unsigned long long t =
      (unsigned long long)(getenv("DSACT_DP_TIMEOUT_MS") ? atoll(getenv("DSACT_DP_TIMEOUT_MS")) : 10000) * 1000000ull;
  return t;
}
// two-shot gradient exchange (dp_peer.cuh) from 6 ranks up (measured, profiles/r2_scaling_8gpu_box.txt: one-shot is 5 % faster
// at 4 ranks, two-shot 0.6 % faster at 8); DSACT_DP_TWO_SHOT=0/1 overrides
// DSACT_DP_SPLIT=1: the critics' part of the gradient exchange and of the update on the side branch, beside the policy
// backward (SURVEY.md 8e's overlap).  Validated (replicas bit-identical, tests green in both exchange variants) but not
// faster: 2 ranks one-shot 8637 / 8498 vs 8517 / 8505 steps/s, two-shot 7853 vs 8210 (profiles/r2_ab_dp_split.txt) — the
// data-parallel overhead is barrier skew and launch count, which a second exchange adds to.  Default: one exchange.
static bool dp_split_enabled() {
  static const bool on = getenv("DSACT_DP_SPLIT") && getenv("DSACT_DP_SPLIT")[0] == '1';
  return on;
}
static bool dp_two_shot(const dsact_handle* h) {
  static const char* e = getenv("DSACT_DP_TWO_SHOT");
  if (e && (e[0] == '0' || e[0] == '1')) return e[0] == '1';
  return h->dp.world >= 6;
}
static long long dp_npad(const dsact_handle* h) { return (2 * h->q.n + h->pi.n + 1 + 3) / 4 * 4; }
// `part`: 0 = the whole buffer, 1 = the critics' groups [0, n_q2 / 4) (kind-4 flags), 2 = the rest (kind-2 flags)
static void enqueue_dp_reduce_scatter(dsact_handle* h, Ctx& c, int part = 0) {
  const long long g_all = dp_npad(h) / 4, g_q = (2 * h->q.n) / 4;
  const long long G0 = part == 2 ? g_q : 0, G1 = part == 1 ? g_q : g_all;
  const long long groups = G1 - G0, per = (groups + h->dp.world - 1) / h->dp.world;
  DpSlice sl;
  sl.g_lo = G0 + per * h->dp.rank;
  sl.g_hi = sl.g_lo + per < G1 ? sl.g_lo + per : G1;
  if (sl.g_lo > G1) sl.g_lo = G1;
  sl.red_off = DP_GRADS_OFF + dp_npad(h);
  sl.ticket = reinterpret_cast<int*>(h->dp_buf) + DP_TICKET + (part == 1 ? 1 : 0);   // block ticket of this launch
  sl.flag_kind = part == 1 ? 4 : 2;
  int blocks = (int)((per + 255) / 256); if (blocks < 1) blocks = 1; if (blocks > 2 * h->num_sms) blocks = 2 * h->num_sms;
  launch_k(dp_reduce_scatter_kernel, blocks, 256, 0, c, h->dp, sl, (const float*)h->buf.state);
  c.done();
}

// One exchange of the peer-memory data-parallel path (dp_peer.cuh): kind 0 = critic-std sums, 1 = logged sums.
static void enqueue_dp_exchange(dsact_handle* h, int kind, Ctx& c) {
  launch_k(dp_exchange_kernel, 1, 32 * h->dp.world, 0, c, h->dp, h->buf.state, kind, dp_timeout_ns());
  c.done();
}

// `dp_std_exchange`: the std sums are complete once sample_kernel has run, one whole forward chain before the loss needs
// them: in a captured step their exchange (kernel + NVLink flag round trip + whatever the ranks are skewed by) runs as a
// side branch under that chain.
static void enqueue_phase1(dsact_handle* h, const dsact_batch& bt, const dsact_noise* nz, Ctx& c, bool inputs_imaged = false,
                           bool prologue_forked = false, bool dp_std_exchange = false) {
  const dsact_config& cf = h->cfg;
  const Net &q = h->q, &pi = h->pi;
  const Arena& ar = h->ar;
  float* W = h->W();
  const int B = bt.batch, O = cf.obs_dim, A = cf.act_dim;
  float* P = h->buf.params;
  float* T = h->buf.targets;
  const float* Qb[4] = {P, P + q.n, T, T + q.n};        // q1, q2, q1', q2'
  const float* PIb[2] = {P + 2 * q.n, T + 2 * q.n};     // pi, pi'
  auto ten = [&](const float* f, const ImgSlot& s) { Ten t; t.f = const_cast<float*>(f); t.im = h->img(s, B); return t; };
  const ImgSlot none;

  if (prologue_forked) {
    cudaStreamWaitEvent(c.s, h->ev_pro_join, 0);
  } else {
    enqueue_prologue(h, bt, nz, c, inputs_imaged);
  }

  const float *eps1, *eps2, *z3, *z4;
  if (nz) { eps1 = nz->eps1; eps2 = nz->eps2; z3 = nz->z3; z4 = nz->z4; }
  else {
    eps1 = W + ar.eps1; eps2 = W + ar.eps2; z3 = W + ar.z3; z4 = W + ar.z4;   // sample_kernel steps the counter
  }

  const Ten t_obs = ten(bt.obs, ar.i_obs), t_obs2 = ten(bt.obs2, ar.i_obs2), t_act = ten(bt.act, ar.i_act);
  const Ten t_none;

  const bool fused = h->fused();
  const Img i_none;
  if (fused) {  // wave A as ONE launch: each CTA runs a 128-row block through every layer of its pass
    ChainBuild cb(h->passes());
    chain_fwd_pass(cb, h, pi, PIb[0], ar.i_wpi[0], t_obs.im, O, i_none, 0, 0, B, cf.act_pi, ar.zP, ar.i_hP, W + ar.logitsP);
    chain_fwd_pass(cb, h, pi, PIb[1], ar.i_wpi[1], t_obs2.im, O, i_none, 0, 0, B, cf.act_pi, nullptr, nullptr, W + ar.logitsT);
    for (int k = 0; k < 2; ++k)
      chain_fwd_pass(cb, h, q, Qb[k], ar.i_wq[k], t_obs.im, O, t_act.im, A, ar.kpad_q0, B, cf.act_q, ar.zQ[k], ar.i_hQ[k], W + ar.outQ[k]);
    launch_chain(h, cb, CLS_GEMM_FWD, c);
  }
  // wave A: pi(obs), pi'(obs2), Q1(s,a), Q2(s,a), layer by layer
  const int depth = fused ? 0 : (pi.L > q.L ? pi.L : q.L) + 1;
  for (int j = 0; j < depth; ++j) {
    Group G;
    if (j <= pi.L) {
      const Ten inP = j == 0 ? t_obs : ten(W + ar.hP[j - 1], ar.i_hP[j - 1]);
      const Ten inT = j == 0 ? t_obs2 : ten(W + ar.hT[j - 1], ar.i_hT[j - 1]);
      const Ten outP = j == pi.L ? ten(W + ar.logitsP, none) : ten(W + ar.hP[j], ar.i_hP[j]);
      const Ten outT = j == pi.L ? ten(W + ar.logitsT, none) : ten(W + ar.hT[j], ar.i_hT[j]);
      add_fwd(G, pi, j, weight(h, pi, PIb[0], j, ar.i_wpi[0][j]), inP, pi.s[j], t_none, 0, 0, outP, j == pi.L ? nullptr : W + ar.zP[j], B, cf.act_pi);
      add_fwd(G, pi, j, weight(h, pi, PIb[1], j, ar.i_wpi[1][j]), inT, pi.s[j], t_none, 0, 0, outT, nullptr, B, cf.act_pi);
    }
    if (j <= q.L) {
      for (int k = 0; k < 2; ++k) {
        const Ten out = j == q.L ? ten(W + ar.outQ[k], none) : ten(W + ar.hQ[k][j], ar.i_hQ[k][j]);
        float* z = j == q.L ? nullptr : W + ar.zQ[k][j];
        const Wt w = weight(h, q, Qb[k], j, ar.i_wq[k][j]);
        if (j == 0) add_fwd(G, q, 0, w, t_obs, O, t_act, A, ar.kpad_q0, out, z, B, cf.act_q);
        else add_fwd(G, q, j, w, ten(W + ar.hQ[k][j - 1], ar.i_hQ[k][j - 1]), q.s[j], t_none, 0, 0, out, z, B, cf.act_q);
      }
    }
    launch_group(h, G, V_FWD, c);
  }

  // rsample of both policies (utils/act_distribution_cls.py:44-54)
  {
    SampleArgs a;
    a.logits[0] = W + ar.logitsP; a.logits[1] = W + ar.logitsT;
    a.eps[0] = eps1; a.eps[1] = eps2;
    a.act[0] = W + ar.new_act; a.act[1] = W + ar.act2;
    a.logp[0] = W + ar.logp_new; a.logp[1] = W + ar.logp2;
    a.hi = h->buf.act_high; a.lo = h->buf.act_low; a.state = h->buf.state;
    a.B = B; a.A = A; a.min_log_std = (float)cf.min_log_std; a.max_log_std = (float)cf.max_log_std; a.gauss = cf.act_dist;
    a.img[0] = img_out(h, ar.i_new_act); a.img[1] = img_out(h, ar.i_act2);
    a.out_q[0] = W + ar.outQ[0]; a.out_q[1] = W + ar.outQ[1];
    a.advance_rng = nz ? 0 : 1;
    int blocks = (B + 7) / 8; if (blocks > 4 * h->num_sms) blocks = 4 * h->num_sms;
    launch_k(sample_kernel, dim3(blocks, 2), 256, 0, c, a); c.done();
  }
  bool dp_forked = false;
  if (dp_std_exchange) {
    if (c.side) {
      cudaEventRecord(h->ev_dp_fork, c.s);
      cudaStreamWaitEvent(c.side, h->ev_dp_fork, 0);
      Ctx cs{c.side, 0, cudaSuccess};
      cs.pdl = c.pdl;
      enqueue_dp_exchange(h, 0, cs);
      cudaEventRecord(h->ev_dp_join, c.side);
      c.launches += cs.launches;
      if (cs.err != cudaSuccess && c.err == cudaSuccess) c.err = cs.err;
      dp_forked = true;
    } else {
      enqueue_dp_exchange(h, 0, c);
    }
  }

  // wave B: Q1', Q2' on (s', a') and Q1, Q2 on (s, a~)
  const Ten t_new_act = ten(W + ar.new_act, ar.i_new_act), t_act2 = ten(W + ar.act2, ar.i_act2);
  if (fused) {
    ChainBuild cb(h->passes());
    for (int k = 0; k < 2; ++k)
      chain_fwd_pass(cb, h, q, Qb[2 + k], ar.i_wq[2 + k], t_obs2.im, O, t_act2.im, A, ar.kpad_q0, B, cf.act_q, nullptr, nullptr, W + ar.outQ[2 + k]);
    for (int k = 0; k < 2; ++k)
      chain_fwd_pass(cb, h, q, Qb[k], ar.i_wq[k], t_obs.im, O, t_new_act.im, A, ar.kpad_q0, B, cf.act_q, ar.zQ[4 + k], nullptr, W + ar.outQ[4 + k]);
    launch_chain(h, cb, CLS_GEMM_FWD, c);
  }
  for (int j = 0; j <= (fused ? -1 : q.L); ++j) {
    Group G;
    for (int p = 2; p < 6; ++p) {
      const int k = p & 1;
      const bool tgt = p < 4;
      const int wn = tgt ? 2 + k : k;
      const Ten out = j == q.L ? ten(W + ar.outQ[p], none) : ten(W + ar.hQ[p][j], ar.i_hQ[p][j]);
      float* z = (j == q.L || tgt) ? nullptr : W + ar.zQ[p][j];
      const Wt w = weight(h, q, Qb[wn], j, ar.i_wq[wn][j]);
      if (j == 0) add_fwd(G, q, 0, w, tgt ? t_obs2 : t_obs, O, tgt ? t_act2 : t_new_act, A, ar.kpad_q0, out, z, B, cf.act_q);
      else add_fwd(G, q, j, w, ten(W + ar.hQ[p][j - 1], ar.i_hQ[p][j - 1]), q.s[j], t_none, 0, 0, out, z, B, cf.act_q);
    }
    launch_group(h, G, V_FWD, c);
  }

  if (dp_forked) cudaStreamWaitEvent(c.s, h->ev_dp_join, 0);
  h->pending_eps1 = eps1; h->pending_z3 = z3; h->pending_z4 = z4;
  c.check();
}

// `defer_reduce`: the caller enqueues enqueue_apply(.., reduce_slabs = true) next, which folds the split slabs itself
static bool slabs_foldable(const dsact_handle* h) {
  return h->tc() && ((uintptr_t)(h->W() + h->ar.slabs) & 15) == 0 && ((uintptr_t)h->buf.grads & 15) == 0;
}
enum { REDUCE_INPLACE = 0, REDUCE_DEFER = 1, REDUCE_DP = 2 };   // where the weight-gradient slabs get folded
static TailArgs tail_args(const dsact_handle* h, int64_t global_batch, int rows, bool enabled) {
  const Net &q = h->q, &pi = h->pi;
  TailArgs t;
  t.sc.tau_b = (float)h->cfg.tau_b; t.sc.alpha_fixed = (float)h->cfg.alpha_fixed;
  t.sc.inv_global_batch = (float)(1.0 / (double)global_batch);
  t.sc.auto_alpha = h->cfg.auto_alpha; t.sc.log_alpha = h->buf.params + 2 * q.n + pi.n;
  t.target_entropy = -(float)h->cfg.act_dim; t.rows = rows; t.enabled = enabled ? 1 : 0;
  return t;
}
// `fold_tail`: the caller's next kernels (dp_grad_fold / apply) do the end-of-backward bookkeeping, no phase2_tail launch
static void enqueue_apply(dsact_handle* h, Ctx& c, bool reduce_slabs, bool dp, const TailArgs* tail, int part);
// `early_apply` (single-GPU fused steps with the folded tail): update the critics on the side branch as soon as their
// weight gradients are complete, beside the policy backward; the caller's enqueue_apply then does the rest.
static void enqueue_phase2(dsact_handle* h, const dsact_batch& bt, int64_t global_batch, Ctx& c, int reduce_mode = REDUCE_INPLACE,
                           bool fold_tail = false, const TailArgs* early_apply = nullptr, bool dp_early = false) {
  const bool defer_reduce = reduce_mode != REDUCE_INPLACE;
  const dsact_config& cf = h->cfg;
  const Net &q = h->q, &pi = h->pi;
  const Arena& ar = h->ar;
  float* W = h->W();
  const int B = bt.batch, O = cf.obs_dim, A = cf.act_dim;
  const bool tc = h->tc();
  float* P = h->buf.params;
  float* G_ = h->buf.grads;
  const float *Pq[2] = {P, P + q.n}, *Ppi = P + 2 * q.n;
  float *Gq[2] = {G_, G_ + q.n}, *Gpi = G_ + 2 * q.n;
  const float invB = (float)(1.0 / (double)global_batch);
  auto ten = [&](const float* f, const ImgSlot& s) { Ten t; t.f = const_cast<float*>(f); t.im = h->img(s, B); return t; };
  const ImgSlot none;

  StepScalars sc;
  sc.tau_b = (float)cf.tau_b; sc.alpha_fixed = (float)cf.alpha_fixed; sc.inv_global_batch = invB;
  sc.auto_alpha = cf.auto_alpha; sc.log_alpha = P + 2 * q.n + pi.n;
  {
    LossArgs a;
    a.sc = sc;
    a.rew = bt.rew; a.done = bt.done;
    a.z3 = h->pending_z3; a.z4 = h->pending_z4;
    a.logp2 = W + ar.logp2; a.logp_new = W + ar.logp_new;
    for (int k = 0; k < 2; ++k) {
      a.out_q[k] = W + ar.outQ[k]; a.out_qt[k] = W + ar.outQ[2 + k]; a.out_qa[k] = W + ar.outQ[4 + k];
      a.d_out_q[k] = W + ar.dOut[k]; a.d_out_qa[k] = W + ar.dOut[4 + k];
      a.gbias_q[k] = Gq[k] + q.b[q.L];
      a.gbias_q_raw[k] = nullptr;
    }
    a.state = h->buf.state; a.B = B; a.gamma = (float)cf.gamma; a.inv_global_batch = invB;
    for (int k = 0; k < 2; ++k) { a.img_q[k] = img_out(h, ar.i_dOut[k]); a.img_qa[k] = img_out(h, ar.i_dOut[4 + k]); }
    int blocks = (B + 63) / 64; if (blocks > 4 * h->num_sms) blocks = 4 * h->num_sms;   // latency bound: spread over the SMs
    launch_k(loss_kernel, blocks, 64, 0, c, a); c.done();
  }
  const int passes[4] = {0, 1, 4, 5};
  const Ten t_obs = ten(bt.obs, ar.i_obs), t_act = ten(bt.act, ar.i_act);

  // wave C: critic passes 0,1 (dgrad + wgrad) and actor passes 4,5 (dgrad only), top layer down.
  // The freeze trick of the reference (dsac_v2.py:166-181) makes the two backward passes independent.  Default: one
  // 4-pass dgrad chain, then the critics' weight gradients as a side branch beside the policy backward.  Opt-in
  // (DSACT_BWD_SPLIT=1): the critics' own backward (dgrad chain 0,1 -> their weight gradients) as a side branch beside
  // the whole actor path (dgrad chain 4,5 -> policy_grad -> policy dgrad chain -> policy weight gradients) — measured
  // 6 us SLOWER per step at B = 4096 (profiles/r2_ab_bwd_split.txt): two half-wave chain launches lose more than the
  // earlier start of the policy path gains.
  Group gw;  // every weight-gradient problem of the two critics
  const bool fused = h->fused();
  static const bool split_on = getenv("DSACT_BWD_SPLIT") && getenv("DSACT_BWD_SPLIT")[0] == '1';
  const bool two_branches = fused && c.side != nullptr && split_on;
  Ctx cs{c.side, 0, cudaSuccess};
  cs.pdl = c.pdl;
  if (two_branches) {
    cudaEventRecord(h->ev_fork, c.s);
    cudaStreamWaitEvent(c.side, h->ev_fork, 0);
  }
  if (fused) {  // dgrad as chain launches: dz stays in tensor memory between layers
    auto chain_of = [&](int pp0, int pp1, Ctx& cx) {
      ChainBuild cb(h->passes());
      for (int pp = pp0; pp < pp1; ++pp) {
        const int p = passes[pp], k = p & 1;
        chain_dgrad_pass(cb, h, q, ar.i_wq[k], h->img(ar.i_dOut[p], B), B, cf.act_q, ar.zQ[p], p < 2 ? Gq[k] : nullptr,
                         p < 2 ? ar.i_dzQ[p] : nullptr, p < 2 ? nullptr : W + ar.dAct[k], ar.kpad_q0, A);
      }
      launch_chain(h, cb, CLS_GEMM_DGRAD, cx);
    };
    if (two_branches) { chain_of(0, 2, cs); chain_of(2, 4, c); }
    else chain_of(0, 4, c);
  }
  for (int j = q.L; j >= 1; --j) {
    Group gd;
    for (int pp = 0; pp < 4; ++pp) {
      const int p = passes[pp], k = p & 1;
      const Ten dY = j == q.L ? ten(W + ar.dOut[p], ar.i_dOut[p]) : ten(W + ar.dzQ[p][j], ar.i_dzQ[p][j]);
      float* gb = p < 2 ? Gq[k] + q.b[j - 1] : nullptr;
      add_dgrad(gd, q, j, weight(h, q, Pq[k], j, ar.i_wq[k][j]), 0, 0, q.s[j], dY, ten(W + ar.dzQ[p][j - 1], ar.i_dzQ[p][j - 1]),
                W + ar.zQ[p][j - 1], gb, B, cf.act_q);
      if (fused) gd.n = gd.g.n = 0;  // done by the chain launch; only the weight-gradient problems are collected here
      if (p < 2) add_wgrad(gw, q, j, Gq[k] + q.w[j], 0, q.s[j], dY, ten(W + ar.hQ[p][j - 1], ar.i_hQ[p][j - 1]), B);
    }
    launch_group(h, gd, V_DGRAD, c);
  }
  {
    Group gd;
    for (int k = 0; k < 2; ++k) {
      const Ten dz0 = ten(W + ar.dzQ[k][0], ar.i_dzQ[k][0]);
      add_wgrad(gw, q, 0, Gq[k] + q.w[0], 0, O, dz0, t_obs, B);
      add_wgrad(gw, q, 0, Gq[k] + q.w[0], O, A, dz0, t_act, B);
      if (!fused)
        add_dgrad(gd, q, 0, weight(h, q, Pq[k], 0, ar.i_wq[k][0]), O, ar.kpad_q0, A, ten(W + ar.dzQ[4 + k][0], ar.i_dzQ[4 + k][0]),
                  ten(W + ar.dAct[k], none), nullptr, nullptr, B, 0);
    }
    if (!two_branches && fused && c.side != nullptr) {   // one 4-pass chain on the main branch, the critics' weight gradients beside the policy backward
      cudaEventRecord(h->ev_fork, c.s);
      cudaStreamWaitEvent(c.side, h->ev_fork, 0);
    }
    if (fused && c.side != nullptr) {
      // the policy backward chain needs ceil(B/128) whole SMs: keep them free of weight-gradient CTAs
      const int chain_ctas = (B + TC_BM - 1) / TC_BM;
      const int cap = h->num_sms - chain_ctas;
      launch_group(h, gw, V_WGRAD, cs, cap >= h->num_sms / 2 ? cap : 0);
      if (early_apply && dp_early) {   // data parallel: the critics' blocks are exchanged and applied here, beside the policy backward
        const long long nq = (2 * q.n) / 4 * 4;   // whole float4 groups of the critics' span
        int blocks = (int)((nq / 4 + 255) / 256); if (blocks > 4 * h->num_sms) blocks = 4 * h->num_sms; if (blocks < 1) blocks = 1;
        TailArgs none; memset(&none, 0, sizeof(none));
        launch_k(dp_grad_fold_kernel, blocks, 256, 0, cs, h->dp_buf + DP_GRADS_OFF, (const float*)G_, (const float*)(W + ar.slabs), nq,
                 ar.nslabs, (long long)ar.slab_stride, (const float*)h->buf.state, none);
        cs.done();
        enqueue_dp_exchange(h, 3, cs);
        if (dp_two_shot(h)) enqueue_dp_reduce_scatter(h, cs, 1);
        enqueue_apply(h, cs, false, true, early_apply, 1);
        h->apply_early = true;
      } else if (early_apply) {   // Adam + Polyak of both critics beside the policy backward: every critic gradient is final here
        enqueue_apply(h, cs, true, false, early_apply, 1);
        h->apply_early = true;
      }
      cudaEventRecord(h->ev_join, c.side);
      c.launches += cs.launches;
      if (cs.err != cudaSuccess && c.err == cudaSuccess) c.err = cs.err;
    } else {
      launch_group(h, gw, V_WGRAD, c);
    }
    launch_group(h, gd, V_DGRAD, c);
    h->join_pending = fused && c.side != nullptr;
  }

  {
    PolicyGradArgs a;
    a.logits = W + ar.logitsP; a.eps = h->pending_eps1; a.d_act1 = W + ar.dAct[0]; a.d_act2 = W + ar.dAct[1];
    a.hi = h->buf.act_high; a.lo = h->buf.act_low;
    a.d_logits = W + ar.dlogits; a.gbias = Gpi + pi.b[pi.L]; a.gbias_ls = nullptr; a.state = h->buf.state;
    a.B = B; a.A = A; a.min_log_std = (float)cf.min_log_std; a.max_log_std = (float)cf.max_log_std; a.gauss = cf.act_dist;
    a.inv_global_batch = invB;
    a.img = img_out(h, ar.i_dlogits);
    a.sc = sc;
    int blocks = (B + 7) / 8; if (blocks > 8 * h->num_sms) blocks = 8 * h->num_sms; if (blocks < 1) blocks = 1;   // a warp per row
    launch_k(policy_grad_kernel, blocks, 256, sizeof(float) * 2 * A, c, a); c.done();
  }

  // wave D: policy backward
  Group gwp;
  if (fused) {
    ChainBuild cb(h->passes());
    chain_dgrad_pass(cb, h, pi, ar.i_wpi[0], h->img(ar.i_dlogits, B), B, cf.act_pi, ar.zP, Gpi, ar.i_dzP, nullptr, 0, 0);
    launch_chain(h, cb, CLS_GEMM_DGRAD, c);
  }
  for (int j = pi.L; j >= 0; --j) {
    const Ten dY = j == pi.L ? ten(W + ar.dlogits, ar.i_dlogits) : ten(W + ar.dzP[j], ar.i_dzP[j]);
    add_wgrad(gwp, pi, j, Gpi + pi.w[j], 0, pi.s[j], dY, j == 0 ? t_obs : ten(W + ar.hP[j - 1], ar.i_hP[j - 1]), B);
    if (j >= 1 && !fused) {
      Group gd;
      add_dgrad(gd, pi, j, weight(h, pi, Ppi, j, ar.i_wpi[0][j]), 0, 0, pi.s[j], dY, ten(W + ar.dzP[j - 1], ar.i_dzP[j - 1]),
                W + ar.zP[j - 1], Gpi + pi.b[j - 1], B, cf.act_pi);
      launch_group(h, gd, V_DGRAD, c);
    }
  }
  launch_group(h, gwp, V_WGRAD, c);

  if (h->join_pending) { cudaStreamWaitEvent(c.s, h->ev_join, 0); h->join_pending = false; }
  if (tc && reduce_mode != REDUCE_DP && !(defer_reduce && slabs_foldable(h))) {  // fold the weight-gradient split slabs into the flat gradient buffer
    const long long n = 2 * q.n + pi.n + 1;
    int blocks = (int)((n + 255) / 256); if (blocks > 4 * h->num_sms) blocks = 4 * h->num_sms;
    launch_k(grad_reduce_kernel, blocks, 256, 0, c, G_, W + ar.slabs, n, ar.nslabs, (long long)ar.slab_stride); c.done();
  }
  AdamHyper hy{cf.lr_q, cf.lr_pi, cf.lr_alpha, cf.adam_beta1, cf.adam_beta2};
  if (!fold_tail) {
    launch_k(phase2_tail_kernel, 1, 32, 0, c, G_ + 2 * q.n + pi.n, h->buf.state, sc, -(float)cf.act_dim, B, hy, defer_reduce ? 1 : 0);
    c.done();
  }
  if (reduce_mode == REDUCE_DP) {  // local total (bias gradients + slabs + log_alpha) -> this rank's block of the exchange buffer
    const long long lo = h->apply_early ? (2 * q.n) / 4 * 4 : 0;   // the critics' groups went out on the side branch
    const long long n = 2 * q.n + pi.n + 1 - lo;
    int blocks = (int)((n / 4 + 255) / 256); if (blocks > 4 * h->num_sms) blocks = 4 * h->num_sms; if (blocks < 1) blocks = 1;
    launch_k(dp_grad_fold_kernel, blocks, 256, 0, c, h->dp_buf + DP_GRADS_OFF + lo, (const float*)G_ + lo, (const float*)(tc ? W + ar.slabs : G_) + lo, n,
             tc ? ar.nslabs : 0, (long long)(tc ? ar.slab_stride : 4), (const float*)h->buf.state, tail_args(h, global_batch, B, fold_tail));
    c.done();
  }
  c.check();
}

static bool fold_tail_enabled() {   // DSACT_FOLD_TAIL=0: keep the separate phase2_tail launch (A/B aid)
  static const bool off = getenv("DSACT_FOLD_TAIL") && getenv("DSACT_FOLD_TAIL")[0] == '0';
  return !off;
}
// `tail` != null: this apply also does the end-of-backward bookkeeping of the step (see TailArgs)
// `part`: 0 = the whole flat buffer; 1 = the critics' span only, without closing the step (launched beside the policy
// backward, see enqueue_phase2); 2 = everything after that span + the end-of-step bookkeeping
static bool apply_split_enabled() {   // DSACT_APPLY_SPLIT=0: one apply launch after the whole backward (A/B aid)
  static const bool off = getenv("DSACT_APPLY_SPLIT") && getenv("DSACT_APPLY_SPLIT")[0] == '0';
  return !off;
}
static void enqueue_apply(dsact_handle* h, Ctx& c, bool reduce_slabs = false, bool dp = false, const TailArgs* tail = nullptr, int part = 0) {
  const dsact_config& cf = h->cfg;
  if (part == 0 && h->apply_early) { part = 2; h->apply_early = false; }   // phase 2 already updated the critics
  ApplyArgs a;
  a.params = h->buf.params; a.targets = h->buf.targets; a.grads = h->buf.grads; a.m = h->buf.adam_m; a.v = h->buf.adam_v;
  a.state = h->buf.state;
  a.n_q2 = 2 * h->q.n; a.n_all = 2 * h->q.n + h->pi.n + 1;
  a.delay_update = cf.delay_update; a.auto_alpha = cf.auto_alpha;
  a.hy = AdamHyper{cf.lr_q, cf.lr_pi, cf.lr_alpha, cf.adam_beta1, cf.adam_beta2};
  a.scalars_ready = (reduce_slabs || dp) ? 1 : 0;   // single-call steps: the phase-2 tail of this very step computed them
  memset(&a.tail, 0, sizeof(a.tail));
  if (tail && tail->enabled) { a.tail = *tail; a.scalars_ready = 2; }   // folded tail: scalars precomputed by the previous apply if stamped
  a.dp_world = 0;
  a.dp_own = nullptr; a.dp_wait_world = 0; a.dp_timeout_ns = dp_timeout_ns();
  for (int r = 0; r < 8; ++r) a.dp_grads[r] = nullptr;
  a.dp_wait_kind = part == 1 ? 4 : 2;
  if (dp && dp_two_shot(h)) {   // the reduced block in this rank's own memory, once every rank's kind-2 (kind-4) flag is here
    a.dp_world = 1;
    a.dp_grads[0] = h->dp_buf + DP_GRADS_OFF + dp_npad(h);
    a.dp_own = h->dp_buf; a.dp_wait_world = h->dp.world;
  } else if (dp) {
    a.dp_world = h->dp.world;
    for (int r = 0; r < h->dp.world; ++r) a.dp_grads[r] = h->dp.peer[r] + DP_GRADS_OFF;
  }
  a.eps = (float)cf.adam_eps; a.tau = (float)cf.tau;
  a.omb1 = (float)(1.0 - cf.adam_beta1); a.b2f = (float)cf.adam_beta2; a.omb2 = (float)(1.0 - cf.adam_beta2);
  a.slabs = nullptr; a.nslabs = 0; a.slab_stride = 0;
  if (reduce_slabs && !dp && slabs_foldable(h)) { a.slabs = h->W() + h->ar.slabs; a.nslabs = h->ar.nslabs; a.slab_stride = h->ar.slab_stride; }
  const int64_t g_all = (a.n_all + 3) / 4, g_q = a.n_q2 / 4;   // a group straddling the critic / policy boundary goes with part 2
  a.g_lo = part == 2 ? g_q : 0; a.g_hi = part == 1 ? g_q : g_all; a.finish = part == 1 ? 0 : 1;
  a.next_scalars = (h->tc() && prologue_merged()) ? 0 : 1;   // the merged prologue of every step forms them itself
  int blocks = (int)((a.g_hi - a.g_lo + 255) / 256);   // one 4-element group per thread
  if (blocks > 8 * h->num_sms) blocks = 8 * h->num_sms;
  if (blocks < 1) blocks = 1;
  // (its last block also advances the step counters)
  if (a.dp_world > 0) launch_k(apply_kernel<2>, blocks, 256, 0, c, a);
  else if (a.nslabs > 0) launch_k(apply_kernel<1>, blocks, 256, 0, c, a);
  else launch_k(apply_kernel<0>, blocks, 256, 0, c, a);
  c.done();
  c.check();
}

// `images_only`: the caller is a fused tcgen05 step, which reads obs / obs2 / act through their bf16 images alone
static void enqueue_gather(dsact_handle* h, int B, const int64_t* idx, Ctx& c, bool images_only = false) {
  const Arena& ar = h->ar;
  float* W = h->W();
  // no index list: every warp of the gather draws its row's index itself (the sequence index_kernel defines) and records it
  int64_t* draw = idx ? nullptr : reinterpret_cast<int64_t*>(W + ar.idx);
  int blocks = (B + 7) / 8; if (blocks > 8 * h->num_sms) blocks = 8 * h->num_sms;
  launch_k(gather_kernel, blocks, 256, 0, c, h->rb.obs, h->rb.obs2, h->rb.act, h->rb.rew, h->rb.done, h->rb.logp, idx,
                                          W + ar.obs, W + ar.obs2, W + ar.act, W + ar.rew, W + ar.done, W + ar.logp, B,
                                          h->cfg.obs_dim, h->cfg.act_dim, img_out(h, ar.i_obs), img_out(h, ar.i_obs2), img_out(h, ar.i_act),
                                          draw, (unsigned long long)h->seed, (const float*)h->buf.state, images_only ? 0 : 1);
  c.done();
  c.check();
}

// ---- graph cache -------------------------------------------------------------
enum { K_STEP = 1, K_PHASE1 = 2, K_PHASE2 = 3, K_APPLY = 4, K_GRADS = 5, K_SAMPLE = 6, K_REPLAY_STEP = 7, K_DP_STEP = 8, K_DP_REPLAY_STEP = 9 };

static void drop_graphs(dsact_handle* h) {
  for (auto& e : h->graphs) cudaGraphExecDestroy(e.exec);
  h->graphs.clear();
}

template <typename F>
static int run(dsact_handle* h, cudaStream_t user, const GraphKey& key, F enqueue) {
  if (!h->cfg.use_graph) {
    Ctx c{user, 0, cudaSuccess};
    c.pdl = h->tc();
    enqueue(c);
    if (c.err != cudaSuccess) return fail(DSACT_ECUDA, "kernel launch failed: %s", cudaGetErrorString(c.err));
    h->launches += c.launches;
    h->last_launches = c.launches;
    return DSACT_OK;
  }
  GraphEntry* hit = nullptr;
  for (auto& e : h->graphs)
    if (e.key == key) { hit = &e; break; }
  if (!hit) {
    CUDA_TRY(cudaStreamBeginCapture(h->cap_stream, cudaStreamCaptureModeRelaxed));
    Ctx c{h->cap_stream, 0, cudaSuccess};
    c.pdl = h->tc();
    c.side = h->side_stream;
    enqueue(c);
    cudaGraph_t graph = nullptr;
    cudaError_t e = cudaStreamEndCapture(h->cap_stream, &graph);
    if (c.err != cudaSuccess || e != cudaSuccess) {
      if (graph) cudaGraphDestroy(graph);
      return fail(DSACT_ECUDA, "graph capture failed: %s", cudaGetErrorString(c.err != cudaSuccess ? c.err : e));
    }
    cudaGraphExec_t exec = nullptr;
    e = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    if (e != cudaSuccess) return fail(DSACT_ECUDA, "cudaGraphInstantiate failed: %s", cudaGetErrorString(e));
    if (h->graphs.size() >= 16) {  // evict the least recently used
      size_t victim = 0;
      for (size_t i = 1; i < h->graphs.size(); ++i)
        if (h->graphs[i].stamp < h->graphs[victim].stamp) victim = i;
      cudaGraphExecDestroy(h->graphs[victim].exec);
      h->graphs.erase(h->graphs.begin() + victim);
    }
    h->graphs.push_back(GraphEntry{key, exec, c.launches, 0});
    hit = &h->graphs.back();
  }
  hit->stamp = ++h->stamp;
  CUDA_TRY(cudaGraphLaunch(hit->exec, user));
  h->launches += hit->launches;
  h->last_launches = hit->launches;
  return DSACT_OK;
}

static GraphKey make_key(int kind, const dsact_batch* b, const dsact_noise* n, int64_t gb) {
  GraphKey k;
  memset(&k, 0, sizeof(k));
  k.kind = kind;
  if (b) { k.p[0] = b->obs; k.p[1] = b->act; k.p[2] = b->rew; k.p[3] = b->obs2; k.p[4] = b->done; k.batch = b->batch; }
  if (n) { k.p[5] = n->eps1; k.p[6] = n->eps2; k.p[7] = n->z3; k.p[8] = n->z4; }
  k.gb = gb;
  return k;
}

static int check_batch(const dsact_handle* h, const dsact_batch* b) {
  if (!h) return fail(DSACT_EINVAL, "null handle");
  if (!h->bound) return fail(DSACT_ESTATE, "dsact_bind has not been called");
  if (!b || !b->obs || !b->act || !b->rew || !b->obs2 || !b->done) return fail(DSACT_EINVAL, "null batch pointer");
  if (b->batch < 1 || b->batch > h->cfg.max_batch)
    return fail(DSACT_EINVAL, "batch %d outside [1, max_batch=%d]", b->batch, h->cfg.max_batch);
  return DSACT_OK;
}
static int check_noise(const dsact_noise* n) {
  if (n && (!n->eps1 || !n->eps2 || !n->z3 || !n->z4)) return fail(DSACT_EINVAL, "null noise pointer");
  return DSACT_OK;
}

// true when `bt` is the arena minibatch that the preceding dsact_replay_sample gathered (images already there)
static bool take_arena_images(dsact_handle* h, const dsact_batch& bt) {
  const bool yes = h->tc() && h->arena_imaged && bt.obs == h->W() + h->ar.obs && bt.obs2 == h->W() + h->ar.obs2 &&
                   bt.act == h->W() + h->ar.act;
  // any other batch is imaged into the same shared slots by the call that asked: the arena's images are gone after it.
  // (The arena views handed out by dsact_replay_sample are read-only for the same reason: edits are not re-imaged.)
  if (!yes) h->arena_imaged = false;
  return yes;
}

static int sync_iteration(dsact_handle* h, int64_t iteration, cudaStream_t s) {
  if (iteration < 0 || iteration > 0x7fffffff) return fail(DSACT_EINVAL, "iteration out of range");
  if (h->dev_iter != iteration) {
    set_iter_kernel<<<1, 32, 0, s>>>(h->buf.state, (int)iteration);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
  }
  return DSACT_OK;
}

// ---- C ABI ---------------------------------------------------------------------
extern "C" {

const char* dsact_last_error(void) { return g_err; }
int dsact_abi_version(void) { return DSACT_ABI_VERSION; }

static int validate(const dsact_config* c) {
  if (!c) return fail(DSACT_EINVAL, "null config");
  if (c->abi_version != DSACT_ABI_VERSION) return fail(DSACT_EINVAL, "abi_version %d != %d", c->abi_version, DSACT_ABI_VERSION);
  if (c->obs_dim < 1 || c->act_dim < 1) return fail(DSACT_EINVAL, "obs_dim/act_dim must be positive");
  if (c->n_hidden_q < 1 || c->n_hidden_q > DSACT_MAX_HIDDEN || c->n_hidden_pi < 1 || c->n_hidden_pi > DSACT_MAX_HIDDEN)
    return fail(DSACT_EINVAL, "1..%d hidden layers supported", DSACT_MAX_HIDDEN);
  for (int j = 0; j < c->n_hidden_q; ++j) if (c->hidden_q[j] < 1) return fail(DSACT_EINVAL, "bad value hidden size");
  for (int j = 0; j < c->n_hidden_pi; ++j) if (c->hidden_pi[j] < 1) return fail(DSACT_EINVAL, "bad policy hidden size");
  if (c->act_q < 0 || c->act_q > DSACT_ACT_SELU || c->act_pi < 0 || c->act_pi > DSACT_ACT_SELU)
    return fail(DSACT_EINVAL, "unknown activation");
  if (c->max_batch < 1) return fail(DSACT_EINVAL, "max_batch must be positive");
  if (c->delay_update < 1) return fail(DSACT_EINVAL, "delay_update must be >= 1");
  if (c->gemm_mode < DSACT_GEMM_FP32 || c->gemm_mode > DSACT_GEMM_BF16) return fail(DSACT_EINVAL, "unknown gemm_mode %d", c->gemm_mode);
  if (c->act_dist != 0 && c->act_dist != 1) return fail(DSACT_EINVAL, "act_dist must be 0 (TanhGaussDistribution) or 1 (GaussDistribution)");
  return DSACT_OK;
}

int dsact_query_layout(const dsact_config* cfg, dsact_layout* out) {
  int rc = validate(cfg);
  if (rc) return rc;
  if (!out) return fail(DSACT_EINVAL, "null out");
  Net q, pi;
  q.build(cfg->obs_dim + cfg->act_dim, cfg->hidden_q, cfg->n_hidden_q, 2);
  pi.build(cfg->obs_dim, cfg->hidden_pi, cfg->n_hidden_pi, 2 * cfg->act_dim);
  Arena ar;
  ar.build(*cfg, q, pi);
  out->n_q = q.n; out->n_pi = pi.n;
  out->n_params = 2 * q.n + pi.n + 1;
  out->n_targets = 2 * q.n + pi.n;
  out->workspace_bytes = ar.total * (int64_t)sizeof(float);
  out->state_floats = ST_FLOATS;
  out->max_batch = cfg->max_batch;
  return DSACT_OK;
}

int dsact_create(const dsact_config* cfg, int device, dsact_handle** out) {
  int rc = validate(cfg);
  if (rc) return rc;
  if (!out) return fail(DSACT_EINVAL, "null out");
  CUDA_TRY(cudaSetDevice(device));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return fail(DSACT_EARCH, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
  dsact_handle* h = new dsact_handle();
  h->cfg = *cfg;
  h->device = device;
  h->num_sms = prop.multiProcessorCount;
  h->q.build(cfg->obs_dim + cfg->act_dim, cfg->hidden_q, cfg->n_hidden_q, 2);
  h->pi.build(cfg->obs_dim, cfg->hidden_pi, cfg->n_hidden_pi, 2 * cfg->act_dim);
  h->ar.build(*cfg, h->q, h->pi);
  h->bound = h->rb_bound = false;
  h->seed = 0x5DEECE66Dull;
  h->dev_iter = -1;
  h->dev_rb_size = -1;
  h->pending_batch = 0;
  h->arena_imaged = false;
  h->stamp = 0; h->launches = 0; h->last_launches = 0;
  cudaError_t e = cudaStreamCreateWithFlags(&h->cap_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->side_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_pro_fork, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_pro_join, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_dp_fork, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_dp_join, cudaEventDisableTiming);
  if (e != cudaSuccess) { delete h; return fail(DSACT_ECUDA, "cudaStreamCreate failed: %s", cudaGetErrorString(e)); }
  *out = h;
  return DSACT_OK;
}

void dsact_destroy(dsact_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  drop_graphs(h);
  cudaStreamDestroy(h->cap_stream);
  cudaStreamDestroy(h->side_stream);
  cudaEventDestroy(h->ev_fork);
  cudaEventDestroy(h->ev_join);
  cudaEventDestroy(h->ev_pro_fork);
  cudaEventDestroy(h->ev_pro_join);
  cudaEventDestroy(h->ev_dp_fork);
  cudaEventDestroy(h->ev_dp_join);
  for (int r = 0; r < DP_MAX_RANKS; ++r) if (h->dp_opened[r]) cudaIpcCloseMemHandle(h->dp_opened[r]);
  if (h->dp_buf) cudaFree(h->dp_buf);
  for (int t = 0; t < 2; ++t) {
    if (h->stage_buf[t]) cudaFree(h->stage_buf[t]);
    if (h->ev_stage_ready[t]) cudaEventDestroy(h->ev_stage_ready[t]);
    if (h->ev_stage_done[t]) cudaEventDestroy(h->ev_stage_done[t]);
  }
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  delete h;
}

int dsact_bind(dsact_handle* h, const dsact_buffers* b) {
  if (!h || !b) return fail(DSACT_EINVAL, "null argument");
  if (!b->params || !b->targets || !b->grads || !b->adam_m || !b->adam_v || !b->act_high || !b->act_low || !b->state || !b->workspace)
    return fail(DSACT_EINVAL, "null buffer pointer");
  if ((reinterpret_cast<uintptr_t>(b->workspace) & 255) != 0) return fail(DSACT_EINVAL, "workspace must be 256-byte aligned");
  h->buf = *b;
  h->bound = true;
  h->arena_imaged = false;
  if (h->tc()) {  // bias regions of the wgrad slabs are never written by a kernel: they must read as zero
    CUDA_TRY(cudaSetDevice(h->device));
    CUDA_TRY(cudaMemset(h->W() + h->ar.slabs, 0, sizeof(float) * (size_t)h->ar.nslabs * h->ar.slab_stride));
  }
  h->dev_iter = -1;
  h->dev_rb_size = -1;
  drop_graphs(h);
  return DSACT_OK;
}

int dsact_seed(dsact_handle* h, uint64_t seed) {
  if (!h) return fail(DSACT_EINVAL, "null handle");
  h->seed = seed;
  drop_graphs(h);  // the seed is a baked kernel argument
  return DSACT_OK;
}

int dsact_set_carry(dsact_handle* h, float m1, float m2, int64_t tq, int64_t tp, void* stream) {
  if (!h || !h->bound) return fail(DSACT_ESTATE, "not bound");
  CUDA_TRY(cudaSetDevice(h->device));
  set_carry_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(h->buf.state, m1, m2, (int)tq, (int)tp);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  return DSACT_OK;
}

int dsact_grad_phase1(dsact_handle* h, const dsact_batch* batch, const dsact_noise* noise, void* stream) {
  int rc = check_batch(h, batch);
  if (rc || (rc = check_noise(noise))) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  const dsact_batch bt = *batch;
  dsact_noise nz; const dsact_noise* np = nullptr;
  if (noise) { nz = *noise; np = &nz; }
  const bool imaged = take_arena_images(h, bt);
  rc = run(h, (cudaStream_t)stream, make_key(K_PHASE1, &bt, np, imaged ? 1 : 0), [&](Ctx& c) { enqueue_phase1(h, bt, np, c, imaged); });
  if (rc) return rc;
  h->pending = bt;
  h->pending_batch = bt.batch;
  // (a replayed graph does not run enqueue_phase1, so record the noise pointers here as well)
  h->pending_eps1 = np ? np->eps1 : h->W() + h->ar.eps1;
  h->pending_z3 = np ? np->z3 : h->W() + h->ar.z3;
  h->pending_z4 = np ? np->z4 : h->W() + h->ar.z4;
  return DSACT_OK;
}

int dsact_grad_phase2(dsact_handle* h, int64_t global_batch, void* stream) {
  if (!h || !h->bound) return fail(DSACT_ESTATE, "not bound");
  if (h->pending_batch < 1) return fail(DSACT_ESTATE, "dsact_grad_phase2 without a preceding dsact_grad_phase1");
  if (global_batch < h->pending_batch) return fail(DSACT_EINVAL, "global_batch %lld < local batch %d", (long long)global_batch, h->pending_batch);
  CUDA_TRY(cudaSetDevice(h->device));
  const dsact_batch bt = h->pending;
  dsact_noise nz{h->pending_eps1, nullptr, h->pending_z3, h->pending_z4};
  GraphKey key = make_key(K_PHASE2, &bt, &nz, global_batch);
  return run(h, (cudaStream_t)stream, key, [&](Ctx& c) { enqueue_phase2(h, bt, global_batch, c); });
}

int dsact_compute_grads(dsact_handle* h, const dsact_batch* batch, const dsact_noise* noise, void* stream) {
  int rc = check_batch(h, batch);
  if (rc || (rc = check_noise(noise))) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  const dsact_batch bt = *batch;
  dsact_noise nz; const dsact_noise* np = nullptr;
  if (noise) { nz = *noise; np = &nz; }
  const bool imaged = take_arena_images(h, bt);
  GraphKey gkey = make_key(K_GRADS, &bt, np, bt.batch);
  gkey.size = imaged ? 1 : 0;
  rc = run(h, (cudaStream_t)stream, gkey, [&](Ctx& c) {
    enqueue_phase1(h, bt, np, c, imaged);
    enqueue_phase2(h, bt, bt.batch, c);
  });
  if (rc) return rc;
  h->pending = bt; h->pending_batch = bt.batch;
  return DSACT_OK;
}

int dsact_apply(dsact_handle* h, int64_t iteration, void* stream) {
  if (!h || !h->bound) return fail(DSACT_ESTATE, "not bound");
  CUDA_TRY(cudaSetDevice(h->device));
  int rc = sync_iteration(h, iteration, (cudaStream_t)stream);
  if (rc) return rc;
  rc = run(h, (cudaStream_t)stream, make_key(K_APPLY, nullptr, nullptr, 0), [&](Ctx& c) { enqueue_apply(h, c); });
  if (rc) return rc;
  h->dev_iter = iteration + 1;
  return DSACT_OK;
}

int dsact_step(dsact_handle* h, const dsact_batch* batch, const dsact_noise* noise, int64_t iteration, void* stream) {
  int rc = check_batch(h, batch);
  if (rc || (rc = check_noise(noise))) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  rc = sync_iteration(h, iteration, (cudaStream_t)stream);
  if (rc) return rc;
  const dsact_batch bt = *batch;
  dsact_noise nz; const dsact_noise* np = nullptr;
  if (noise) { nz = *noise; np = &nz; }
  const bool imaged = take_arena_images(h, bt);
  GraphKey skey = make_key(K_STEP, &bt, np, bt.batch);
  skey.size = imaged ? 1 : 0;
  rc = run(h, (cudaStream_t)stream, skey, [&](Ctx& c) {
    enqueue_phase1(h, bt, np, c, imaged);
    const TailArgs ta = tail_args(h, bt.batch, bt.batch, fold_tail_enabled());
    const bool early = ta.enabled && h->fused() && slabs_foldable(h) && apply_split_enabled();
    enqueue_phase2(h, bt, bt.batch, c, REDUCE_DEFER, ta.enabled, early ? &ta : nullptr);
    enqueue_apply(h, c, true, false, &ta);
  });
  if (rc) return rc;
  h->pending = bt; h->pending_batch = bt.batch;
  h->dev_iter = iteration + 1;
  return DSACT_OK;
}

// ---- host minibatches: staging on a private copy stream -------------------------------------------------------
int dsact_stage_host(dsact_handle* h, const dsact_batch* host, dsact_batch* dev, void* stream) {
  int rc = check_batch(h, host);
  if (rc) return rc;
  if (!dev) return fail(DSACT_EINVAL, "null out");
  CUDA_TRY(cudaSetDevice(h->device));
  const int64_t O = h->cfg.obs_dim, A = h->cfg.act_dim, Bm = h->cfg.max_batch;
  const int64_t seg[5] = {round64(Bm * O), round64(Bm * A), round64(Bm), round64(Bm * O), round64(Bm)};   // obs act rew obs2 done
  if (!h->copy_stream) {
    h->stage_floats = seg[0] + seg[1] + seg[2] + seg[3] + seg[4];
    CUDA_TRY(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    for (int t = 0; t < 2; ++t) {
      CUDA_TRY(cudaMalloc(&h->stage_buf[t], sizeof(float) * (size_t)h->stage_floats));
      CUDA_TRY(cudaEventCreateWithFlags(&h->ev_stage_ready[t], cudaEventDisableTiming));
      CUDA_TRY(cudaEventCreateWithFlags(&h->ev_stage_done[t], cudaEventDisableTiming));
    }
  }
  const int t = h->stage_turn;
  const int64_t B = host->batch;
  float* base = h->stage_buf[t];
  float* d_obs = base; float* d_act = d_obs + seg[0]; float* d_rew = d_act + seg[1]; float* d_obs2 = d_rew + seg[2]; float* d_done = d_obs2 + seg[3];
  if (h->stage_done_valid[t]) CUDA_TRY(cudaStreamWaitEvent(h->copy_stream, h->ev_stage_done[t], 0));   // last reader of this set
  CUDA_TRY(cudaMemcpyAsync(d_obs, host->obs, sizeof(float) * B * O, cudaMemcpyHostToDevice, h->copy_stream));
  CUDA_TRY(cudaMemcpyAsync(d_obs2, host->obs2, sizeof(float) * B * O, cudaMemcpyHostToDevice, h->copy_stream));
  CUDA_TRY(cudaMemcpyAsync(d_act, host->act, sizeof(float) * B * A, cudaMemcpyHostToDevice, h->copy_stream));
  CUDA_TRY(cudaMemcpyAsync(d_rew, host->rew, sizeof(float) * B, cudaMemcpyHostToDevice, h->copy_stream));
  CUDA_TRY(cudaMemcpyAsync(d_done, host->done, sizeof(float) * B, cudaMemcpyHostToDevice, h->copy_stream));
  CUDA_TRY(cudaEventRecord(h->ev_stage_ready[t], h->copy_stream));
  CUDA_TRY(cudaStreamWaitEvent((cudaStream_t)stream, h->ev_stage_ready[t], 0));
  dev->obs = d_obs; dev->act = d_act; dev->rew = d_rew; dev->obs2 = d_obs2; dev->done = d_done; dev->logp = nullptr;
  dev->batch = host->batch;
  h->stage_held = t;
  h->stage_turn = t ^ 1;
  return DSACT_OK;
}

int dsact_stage_release(dsact_handle* h, void* stream) {
  if (!h) return fail(DSACT_EINVAL, "null handle");
  if (h->stage_held < 0) return DSACT_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaEventRecord(h->ev_stage_done[h->stage_held], (cudaStream_t)stream));
  h->stage_done_valid[h->stage_held] = true;
  h->stage_held = -1;
  return DSACT_OK;
}

int dsact_step_host(dsact_handle* h, const dsact_batch* host, const dsact_noise* noise, int64_t iteration, void* stream) {
  dsact_batch dev;
  int rc = dsact_stage_host(h, host, &dev, stream);
  if (rc) return rc;
  rc = dsact_step(h, &dev, noise, iteration, stream);
  const int rc2 = dsact_stage_release(h, stream);
  return rc ? rc : rc2;
}

int dsact_read_stats(dsact_handle* h, int64_t global_batch, float* host_out, void* stream) {
  if (!h || !h->bound) return fail(DSACT_ESTATE, "not bound");
  if (!host_out || global_batch < 1) return fail(DSACT_EINVAL, "bad argument");
  CUDA_TRY(cudaSetDevice(h->device));
  const float invB = (float)(1.0 / (double)global_batch);
  const float invBA = (float)(1.0 / ((double)global_batch * h->cfg.act_dim));
  finalize_stats_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(h->buf.state, invB, invBA);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  CUDA_TRY(cudaMemcpyAsync(host_out, h->buf.state + ST_STATS, DSACT_NUM_STATS * sizeof(float), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  return DSACT_OK;
}

// ---- replay ring buffer ----------------------------------------------------------
int dsact_replay_bind(dsact_handle* h, const dsact_replay* rb) {
  if (!h || !rb) return fail(DSACT_EINVAL, "null argument");
  if (!rb->obs || !rb->obs2 || !rb->act || !rb->rew || !rb->done || !rb->logp || rb->capacity < 1)
    return fail(DSACT_EINVAL, "bad replay buffers");
  h->rb = *rb;
  h->rb_bound = true;
  drop_graphs(h);
  return DSACT_OK;
}

int dsact_replay_add(dsact_handle* h, const float* obs, const float* obs2, const float* act, const float* rew,
                     const float* done, const float* logp, int64_t n, int64_t ptr, void* stream) {
  if (!h || !h->rb_bound) return fail(DSACT_ESTATE, "replay buffer not bound");
  if (n < 0 || n > h->rb.capacity || ptr < 0 || ptr >= h->rb.capacity) return fail(DSACT_EINVAL, "bad n/ptr");
  if (n == 0) return DSACT_OK;
  if (!obs || !obs2 || !act || !rew || !done || !logp) return fail(DSACT_EINVAL, "null staging pointer");
  CUDA_TRY(cudaSetDevice(h->device));
  const int64_t first = (ptr + n <= h->rb.capacity) ? n : h->rb.capacity - ptr;
  const int64_t O = h->cfg.obs_dim, A = h->cfg.act_dim;
  struct { float* dst; const float* src; int64_t w; } cols[6] = {
      {h->rb.obs, obs, O}, {h->rb.obs2, obs2, O}, {h->rb.act, act, A}, {h->rb.rew, rew, 1}, {h->rb.done, done, 1}, {h->rb.logp, logp, 1}};
  for (auto& c : cols) {
    CUDA_TRY(cudaMemcpyAsync(c.dst + ptr * c.w, c.src, first * c.w * sizeof(float), cudaMemcpyDefault, (cudaStream_t)stream));
    if (first < n)
      CUDA_TRY(cudaMemcpyAsync(c.dst, c.src + first * c.w, (n - first) * c.w * sizeof(float), cudaMemcpyDefault, (cudaStream_t)stream));
  }
  return DSACT_OK;
}

static int sync_rb_size(dsact_handle* h, int64_t size, cudaStream_t s) {
  if (size < 1 || size > h->rb.capacity) return fail(DSACT_EINVAL, "size %lld outside [1, capacity]", (long long)size);
  if (h->dev_rb_size != size) {
    set_rb_size_kernel<<<1, 32, 0, s>>>(h->buf.state, size);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    h->dev_rb_size = size;
  }
  return DSACT_OK;
}

static dsact_batch arena_batch(const dsact_handle* h, int32_t batch) {
  float* W = h->W();
  dsact_batch b;
  b.obs = W + h->ar.obs; b.act = W + h->ar.act; b.rew = W + h->ar.rew; b.obs2 = W + h->ar.obs2; b.done = W + h->ar.done;
  b.logp = W + h->ar.logp;
  b.batch = batch;
  return b;
}

int dsact_replay_sample(dsact_handle* h, int32_t batch, int64_t size, const int64_t* idx, dsact_batch* out, void* stream) {
  if (!h || !h->bound || !h->rb_bound) return fail(DSACT_ESTATE, "not bound");
  if (batch < 1 || batch > h->cfg.max_batch) return fail(DSACT_EINVAL, "batch outside [1, max_batch]");
  CUDA_TRY(cudaSetDevice(h->device));
  int rc = sync_rb_size(h, size, (cudaStream_t)stream);
  if (rc) return rc;
  GraphKey key = make_key(K_SAMPLE, nullptr, nullptr, 0);
  key.batch = batch; key.idx = idx;
  rc = run(h, (cudaStream_t)stream, key, [&](Ctx& c) {
    enqueue_gather(h, batch, idx, c);
    if (!idx) { launch_k(rng_advance_kernel, 1, 32, 0, c, h->buf.state); c.done(); }
  });
  if (rc) return rc;
  h->arena_imaged = true;
  if (out) *out = arena_batch(h, batch);
  return DSACT_OK;
}

int dsact_replay_step(dsact_handle* h, int32_t batch, int64_t size, const int64_t* idx, const dsact_noise* noise,
                      int64_t iteration, void* stream) {
  if (!h || !h->bound || !h->rb_bound) return fail(DSACT_ESTATE, "not bound");
  if (batch < 1 || batch > h->cfg.max_batch) return fail(DSACT_EINVAL, "batch outside [1, max_batch]");
  int rc = check_noise(noise);
  if (rc) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  if ((rc = sync_rb_size(h, size, (cudaStream_t)stream))) return rc;
  if ((rc = sync_iteration(h, iteration, (cudaStream_t)stream))) return rc;
  const dsact_batch bt = arena_batch(h, batch);
  dsact_noise nz; const dsact_noise* np = nullptr;
  if (noise) { nz = *noise; np = &nz; }
  GraphKey key = make_key(K_REPLAY_STEP, &bt, np, batch);
  key.idx = idx;
  rc = run(h, (cudaStream_t)stream, key, [&](Ctx& c) {
    const bool forked = fork_prologue(h, bt, np, c, true);   // weight images, noise, clears: beside the gather
    enqueue_gather(h, batch, idx, c, h->fused());
    if (!idx && np) { launch_k(rng_advance_kernel, 1, 32, 0, c, h->buf.state); c.done(); }
    enqueue_phase1(h, bt, np, c, true, forked);  // device noise (np == null): phase1 advances the counter after the join
    const TailArgs ta = tail_args(h, batch, batch, fold_tail_enabled());
    const bool early = ta.enabled && h->fused() && slabs_foldable(h) && apply_split_enabled();
    enqueue_phase2(h, bt, batch, c, REDUCE_DEFER, ta.enabled, early ? &ta : nullptr);
    enqueue_apply(h, c, true, false, &ta);
  });
  if (rc) return rc;
  h->pending = bt; h->pending_batch = batch;
  h->arena_imaged = false;   // the arena's images (and, in the fused modes, only they) now belong to this step's gather
  h->dev_iter = iteration + 1;
  return DSACT_OK;
}

// ---- data parallelism over peer memory (dp_peer.cuh) ------------------------------------------------------------
int dsact_dp_export(dsact_handle* h, void* handle_out, int64_t* bytes_out) {
  if (!h || !handle_out) return fail(DSACT_EINVAL, "null argument");
  CUDA_TRY(cudaSetDevice(h->device));
  // header + this rank's gradient block + the reduced block of the two-shot exchange
  const size_t bytes = sizeof(float) * (size_t)(DP_GRADS_OFF + 2 * ((2 * h->q.n + h->pi.n + 1 + 3) / 4 * 4));
  if (!h->dp_buf) {
    CUDA_TRY(cudaMalloc(&h->dp_buf, bytes));
    CUDA_TRY(cudaMemset(h->dp_buf, 0, bytes));
  }
  cudaIpcMemHandle_t ipc;
  CUDA_TRY(cudaIpcGetMemHandle(&ipc, h->dp_buf));
  static_assert(sizeof(ipc) == DSACT_IPC_HANDLE_BYTES, "IPC handle size");
  memcpy(handle_out, &ipc, sizeof(ipc));
  if (bytes_out) *bytes_out = (int64_t)bytes;
  return DSACT_OK;
}

int dsact_dp_connect(dsact_handle* h, int32_t rank, int32_t world, const void* handles) {
  if (!h || !handles) return fail(DSACT_EINVAL, "null argument");
  if (!h->bound) return fail(DSACT_ESTATE, "dsact_bind has not been called");
  if (!h->dp_buf) return fail(DSACT_ESTATE, "dsact_dp_export has not been called");
  if (world < 2 || world > DP_MAX_RANKS || rank < 0 || rank >= world) return fail(DSACT_EINVAL, "rank %d / world %d outside [2, %d]", rank, world, DP_MAX_RANKS);
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaDeviceSynchronize());
  drop_graphs(h);
  for (int r = 0; r < DP_MAX_RANKS; ++r)
    if (h->dp_opened[r]) { cudaIpcCloseMemHandle(h->dp_opened[r]); h->dp_opened[r] = nullptr; }
  h->dp.rank = rank; h->dp.world = world;
  for (int r = 0; r < world; ++r) {
    if (r == rank) { h->dp.peer[r] = h->dp_buf; continue; }
    cudaIpcMemHandle_t ipc;
    memcpy(&ipc, static_cast<const char*>(handles) + (size_t)r * sizeof(ipc), sizeof(ipc));
    void* p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, ipc, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(DSACT_ECUDA, "cudaIpcOpenMemHandle(rank %d): %s", r, cudaGetErrorString(e)); }
    h->dp_opened[r] = p;
    h->dp.peer[r] = static_cast<float*>(p);
  }
  // every rank starts at epoch 0 with clear flags (the caller synchronises the ranks after this call)
  CUDA_TRY(cudaMemset(h->dp_buf, 0, sizeof(float) * DP_GRADS_OFF));
  CUDA_TRY(cudaMemset(h->buf.state + ST_DP_EPOCH, 0, sizeof(float)));
  CUDA_TRY(cudaMemset(h->buf.state + ST_DP_ERR, 0, sizeof(float)));
  CUDA_TRY(cudaDeviceSynchronize());
  h->dp_ready = true;
  return DSACT_OK;
}

// One data-parallel update as one submission: forward, std-sum exchange, losses + backward scaled by 1/global_batch,
// gradient + statistics exchange, Adam on the rank-ordered global sum.  Every rank must call it for the same iteration.
int dsact_dp_step(dsact_handle* h, const dsact_batch* batch, const dsact_noise* noise, int64_t global_batch, int64_t iteration,
                  void* stream) {
  int rc = check_batch(h, batch);
  if (rc || (rc = check_noise(noise))) return rc;
  if (!h->dp_ready) return fail(DSACT_ESTATE, "dsact_dp_connect has not been called");
  if (global_batch < batch->batch) return fail(DSACT_EINVAL, "global_batch %lld < local batch %d", (long long)global_batch, batch->batch);
  CUDA_TRY(cudaSetDevice(h->device));
  if ((rc = sync_iteration(h, iteration, (cudaStream_t)stream))) return rc;
  const dsact_batch bt = *batch;
  dsact_noise nz; const dsact_noise* np = nullptr;
  if (noise) { nz = *noise; np = &nz; }
  const bool imaged = take_arena_images(h, bt);
  GraphKey key = make_key(K_DP_STEP, &bt, np, global_batch);
  key.size = imaged ? 1 : 0;
  rc = run(h, (cudaStream_t)stream, key, [&](Ctx& c) {
    enqueue_phase1(h, bt, np, c, imaged, false, true);
    const TailArgs ta = tail_args(h, global_batch, bt.batch, fold_tail_enabled());
    const bool early = ta.enabled && h->fused() && slabs_foldable(h) && dp_split_enabled();
    enqueue_phase2(h, bt, global_batch, c, REDUCE_DP, ta.enabled, early ? &ta : nullptr, true);
    const bool split = h->apply_early;   // the critics' part went out (and was applied) beside the policy backward
    enqueue_dp_exchange(h, 1, c);
    if (dp_two_shot(h)) enqueue_dp_reduce_scatter(h, c, split ? 2 : 0);
    enqueue_apply(h, c, false, true, &ta);
  });
  if (rc) return rc;
  h->pending = bt; h->pending_batch = bt.batch;
  h->dev_iter = iteration + 1;
  return DSACT_OK;
}

int dsact_dp_replay_step(dsact_handle* h, int32_t batch, int64_t size, const int64_t* idx, const dsact_noise* noise,
                         int64_t global_batch, int64_t iteration, void* stream) {
  if (!h || !h->bound || !h->rb_bound) return fail(DSACT_ESTATE, "not bound");
  if (!h->dp_ready) return fail(DSACT_ESTATE, "dsact_dp_connect has not been called");
  if (batch < 1 || batch > h->cfg.max_batch) return fail(DSACT_EINVAL, "batch outside [1, max_batch]");
  if (global_batch < batch) return fail(DSACT_EINVAL, "global_batch %lld < local batch %d", (long long)global_batch, batch);
  int rc = check_noise(noise);
  if (rc) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  if ((rc = sync_rb_size(h, size, (cudaStream_t)stream))) return rc;
  if ((rc = sync_iteration(h, iteration, (cudaStream_t)stream))) return rc;
  const dsact_batch bt = arena_batch(h, batch);
  dsact_noise nz; const dsact_noise* np = nullptr;
  if (noise) { nz = *noise; np = &nz; }
  GraphKey key = make_key(K_DP_REPLAY_STEP, &bt, np, global_batch);
  key.idx = idx;
  rc = run(h, (cudaStream_t)stream, key, [&](Ctx& c) {
    const bool forked = fork_prologue(h, bt, np, c, true);
    enqueue_gather(h, batch, idx, c, h->fused());
    if (!idx && np) { launch_k(rng_advance_kernel, 1, 32, 0, c, h->buf.state); c.done(); }
    enqueue_phase1(h, bt, np, c, true, forked, true);
    const TailArgs ta = tail_args(h, global_batch, bt.batch, fold_tail_enabled());
    const bool early = ta.enabled && h->fused() && slabs_foldable(h) && dp_split_enabled();
    enqueue_phase2(h, bt, global_batch, c, REDUCE_DP, ta.enabled, early ? &ta : nullptr, true);
    const bool split = h->apply_early;
    enqueue_dp_exchange(h, 1, c);
    if (dp_two_shot(h)) enqueue_dp_reduce_scatter(h, c, split ? 2 : 0);
    enqueue_apply(h, c, false, true, &ta);
  });
  if (rc) return rc;
  h->pending = bt; h->pending_batch = batch;
  h->arena_imaged = false;   // the arena's images (and, in the fused modes, only they) now belong to this step's gather
  h->dev_iter = iteration + 1;
  return DSACT_OK;
}

int dsact_profile_step(dsact_handle* h, const dsact_batch* batch, const dsact_noise* noise, int64_t iteration,
                       void* stream, dsact_profile* out) {
  int rc = check_batch(h, batch);
  if (rc || (rc = check_noise(noise))) return rc;
  if (!out) return fail(DSACT_EINVAL, "null out");
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  rc = sync_iteration(h, iteration, s);
  if (rc) return rc;
  const dsact_batch bt = *batch;
  dsact_noise nz; const dsact_noise* np = nullptr;
  if (noise) { nz = *noise; np = &nz; }
  Prof prof;
  Ctx c{s, 0, cudaSuccess};
  c.pdl = h->tc();
  c.prof = &prof;
  cudaEvent_t e0;
  CUDA_TRY(cudaEventCreate(&e0));
  CUDA_TRY(cudaEventRecord(e0, s));
  enqueue_phase1(h, bt, np, c);
  const TailArgs ta = tail_args(h, bt.batch, bt.batch, fold_tail_enabled());
  enqueue_phase2(h, bt, bt.batch, c, REDUCE_DEFER, ta.enabled);
  enqueue_apply(h, c, true, false, &ta);
  cudaError_t e = cudaStreamSynchronize(s);
  memset(out, 0, sizeof(*out));
  cudaEvent_t prev = e0;
  for (size_t i = 0; i < prof.ev.size(); ++i) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, prev, prof.ev[i]);
    out->ms[prof.cls[i]] += ms;
    out->flops[prof.cls[i]] += prof.flops[i];
    out->launches[prof.cls[i]] += 1;
    out->total_ms += ms;
    prev = prof.ev[i];
  }
  cudaEventDestroy(e0);
  for (auto ev : prof.ev) cudaEventDestroy(ev);
  if (c.err != cudaSuccess || e != cudaSuccess)
    return fail(DSACT_ECUDA, "profile step failed: %s", cudaGetErrorString(c.err != cudaSuccess ? c.err : e));
  h->launches += c.launches;
  h->last_launches = c.launches;
  h->pending = bt; h->pending_batch = bt.batch;
  h->dev_iter = iteration + 1;
  return DSACT_OK;
}

int64_t dsact_launch_count(const dsact_handle* h) { return h ? h->launches : 0; }
int32_t dsact_last_call_launches(const dsact_handle* h) { return h ? h->last_launches : 0; }

int dsact_test_gemm(dsact_handle* h, int32_t variant, const float* A, int32_t lda, const float* B, int32_t ldb,
                    const float* bias, float* C, int32_t ldc, int32_t M, int32_t N, int32_t K, void* stream) {
  if (!h) return fail(DSACT_EINVAL, "null handle");
  if (variant < 0 || variant > 2 || M < 1 || N < 1 || K < 1) return fail(DSACT_EINVAL, "bad argument");
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  Group G;
  GemmProb p = prob_zero();
  p.A[0] = A; p.lda[0] = lda; p.B[0] = B; p.ldb[0] = ldb; p.K[0] = K;
  p.M = M; p.N = N; p.C = C; p.ldc = ldc; p.bias = variant == V_FWD ? bias : nullptr;
  p.epi = variant == V_WGRAD ? EPI_ATOMIC : EPI_STORE;
  G.push(p, TcExtra());
  Ctx c{s, 0, cudaSuccess};
  c.pdl = h->tc();
  void* scratch = nullptr;
  if (h->tc()) {  // test hook only: scratch images (and slabs) come from cudaMalloc, not from the caller
    if (variant == V_WGRAD && ldc != N) return fail(DSACT_EINVAL, "tc wgrad test needs contiguous C");
    const int a_rows = variant == V_WGRAD ? K : M, a_w = variant == V_WGRAD ? M : K;
    const int b_rows = variant == V_FWD ? N : K, b_w = variant == V_FWD ? K : N;
    auto mk = [&](int rows, int w, size_t& off) {
      Img i; i.rows = rows; i.width = w; i.pitch = (w + 7) / 8 * 8; i.plane = round64((int64_t)rows * i.pitch);
      off = (off + 255) / 256 * 256; size_t o = off; off += (size_t)i.plane * 4; i.p = reinterpret_cast<__nv_bfloat16*>(o);
      return i;
    };
    size_t off = 0;
    Img ia = mk(a_rows, a_w, off), ib = mk(b_rows, b_w, off);
    const int nslabs = 4;
    off = (off + 255) / 256 * 256;
    const size_t slab_off = off;
    if (variant == V_WGRAD) off += sizeof(float) * (size_t)nslabs * M * N;
    CUDA_TRY(cudaMalloc(&scratch, off + 256));
    ia.p = reinterpret_cast<__nv_bfloat16*>(reinterpret_cast<uintptr_t>(scratch) + reinterpret_cast<uintptr_t>(ia.p));
    ib.p = reinterpret_cast<__nv_bfloat16*>(reinterpret_cast<uintptr_t>(scratch) + reinterpret_cast<uintptr_t>(ib.p));
    ImgBatch ibt;
    ibt.add(A, lda, ia, a_rows, a_w);
    ibt.add(B, ldb, ib, b_rows, b_w);
    ibt.launch(h, c);
    G.x[0].a[0] = ia; G.x[0].b = ib;
    if (variant == V_WGRAD) {
      G.wg_slab = reinterpret_cast<float*>(reinterpret_cast<uintptr_t>(scratch) + slab_off);
      G.wg_stride = (long long)M * N; G.wg_nslabs = nslabs;
    }
  }
  launch_group(h, G, variant, c);
  if (h->tc() && variant == V_WGRAD && c.err == cudaSuccess) {
    grad_reduce_kernel<<<64, 256, 0, s>>>(C, G.wg_slab, (long long)M * N, G.wg_nslabs, (long long)M * N);
    c.done();
  }
  cudaError_t e = cudaSuccess;
  if (scratch) { e = cudaStreamSynchronize(s); cudaFree(scratch); }
  if (c.err != cudaSuccess || e != cudaSuccess)
    return fail(DSACT_ECUDA, "launch failed: %s", cudaGetErrorString(c.err != cudaSuccess ? c.err : e));
  h->launches += c.launches;
  return DSACT_OK;
}

}  // extern "C"

#include "cnn_engine.cuh"
