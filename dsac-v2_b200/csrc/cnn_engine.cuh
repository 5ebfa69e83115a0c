// DSAC-T update with the reference's CNN approximators (BASELINE config 5; reference networks/cnn.py:30-53 conv stack,
// :151-240 StochaPolicy, :383-461 ActionValueDistri).  Included at the end of engine.cu: it reuses the grouped fp32 GEMM
// launcher, the loss / sample / policy-gradient kernels and apply_kernel of the MLP engine; what is new here is the conv
// stack (conv.cuh) and the two-head wiring (separate `mean` and `log_std` MLPs per network, their outputs packed into the
// [B,2] / [B,2A] arrays the loss kernels read, by strided GEMM outputs).
//
// The same wiring without an encoder (n_conv = 0), with one two-output head per critic (q_heads = 1), with the policy as one
// head / two heads / mean head + learnable log_std row (pi_std) serves the MLP approximators whose variants the tcgen05
// engine does not implement (policy std_type mlp_separated / parameter), and DSAC_V1 (v1_step.cuh).
//
// One eager sequence of launches per step (no graph capture yet):
//   conv forwards: pi(s), pi'(s'), Q1/Q2 features of s (shared by the (s,a) and (s,a~) passes), Q1'/Q2' features of s'
//   heads: pi, pi' -> sample -> Q_k(s,a), Q'_k(s',a'), mean head of Q_k(s,a~) -> loss -> head backward (critics: both
//   heads; actor path: mean head, input gradient only) -> policy_grad -> policy heads backward -> conv backward x3 -> Adam.
// The sequence is enqueued in three parts (phase 1 = every forward, phase 2 = losses + backward, apply = Adam + Polyak)
// that dsact_cnn_step runs back to back and the split entry points (dsact_cnn_grad_phase1/2, _compute_grads, _apply) run
// one at a time, for the gradient-message seam and data-parallel callers.
#pragma once
#include "conv.cuh"

namespace dsact {
__global__ void relu_mask_kernel(float* __restrict__ g, const float* __restrict__ a, long long n) {
  pdl_sync();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    if (!(a[i] > 0.f)) g[i] = 0.f;
}
// logits[b][col0 + j] = row[j]: the learnable log_std row of policy std_type "parameter" broadcast over the batch
// (reference networks/mlp.py:95-96)
__global__ void bcast_row_kernel(float* __restrict__ out, int ld, int col0, const float* __restrict__ row, int B, int A) {
  pdl_sync();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < (long long)B * A; i += (long long)gridDim.x * blockDim.x) {
    const int b = (int)(i / A), j = (int)(i - (long long)b * A);
    out[(size_t)b * ld + col0 + j] = row[j];
  }
}
__global__ void zero_kernel(float* __restrict__ p, long long n) {
  pdl_sync();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) p[i] = 0.f;
}
}  // namespace dsact

struct CnnGeom {   // one network: conv encoder (possibly empty) + 1 or 2 identical head MLPs (+ a learnable log_std row)
  int nconv;
  int nheads;            // 2: separate mean / log_std (std) heads; 1: one head (both outputs, or the mean with a log_std row)
  int64_t ls_row;        // offset of the learnable log_std row [out] (policy std_type "parameter"), or -1
  int C[DSACT_MAX_CONV + 1], H[DSACT_MAX_CONV + 1], W[DSACT_MAX_CONV + 1];   // [0] = input image
  int K[DSACT_MAX_CONV], S[DSACT_MAX_CONV];
  int64_t cw[DSACT_MAX_CONV], cb[DSACT_MAX_CONV];
  int F;                 // flattened feature size
  Net head;              // s[0] = F (+ act_dim), hidden..., s[L+1] = outputs of ONE head
  int64_t head_off[2];   // mean, log_std
  int64_t n;
  bool build(const dsact_cnn_config& c, int extra_in, int out, int heads, bool std_row) {
    nconv = c.n_conv; nheads = heads; ls_row = -1;
    C[0] = c.channels; H[0] = c.height; W[0] = c.width;
    n = 0;
    for (int j = 0; j < nconv; ++j) {
      K[j] = c.conv_kernel[j]; S[j] = c.conv_stride[j];
      C[j + 1] = c.conv_channels[j];
      H[j + 1] = (H[j] - K[j]) / S[j] + 1;
      W[j + 1] = (W[j] - K[j]) / S[j] + 1;
      if (H[j + 1] < 1 || W[j + 1] < 1) return false;
      cw[j] = n; n += (int64_t)C[j + 1] * C[j] * K[j] * K[j];
      cb[j] = n; n += C[j + 1];
    }
    F = C[nconv] * H[nconv] * W[nconv];
    head.build(F + extra_in, c.hidden, c.n_hidden, out);
    if (std_row) { ls_row = n; n += out; }   // nn.Module.parameters() yields a module's own parameters before its children's
    head_off[1] = -1;
    for (int hd = 0; hd < nheads; ++hd) { head_off[hd] = n; n += head.n; }
    return true;
  }
  ConvShape shape(int j, int B) const { return ConvShape{B, C[j], H[j], W[j], C[j + 1], K[j], S[j], H[j + 1], W[j + 1]}; }
  int64_t act_elems(int j) const { return (int64_t)C[j] * H[j] * W[j]; }   // per sample, activation j (0 = image)
};

constexpr int CNN_DGRAD_SMEM = 96 * 1024;   // opt-in dynamic shared memory of conv_dgrad8_kernel

struct CnnHeadBuf { int64_t z[DSACT_MAX_HIDDEN], h[DSACT_MAX_HIDDEN], dz[DSACT_MAX_HIDDEN]; };

struct dsact_cnn_handle {
  dsact_cnn_config cfg;
  int device, num_sms;
  CnnGeom q, pi;
  dsact_buffers buf;
  bool bound = false;
  uint64_t seed = 0x5DEECE66Dull;
  int64_t dev_iter = -1, launches = 0;
  // minibatch and noise of the last dsact_cnn_grad_phase1, read by the dsact_cnn_grad_phase2 that follows it
  dsact_batch pending{};
  int pending_batch = 0;   // 0: no phase 1 awaits its phase 2
  const float *pending_eps1 = nullptr, *pending_z3 = nullptr, *pending_z4 = nullptr;
  // arena (floats from the workspace base)
  int64_t convP[DSACT_MAX_CONV + 1], convT[DSACT_MAX_CONV + 1], convQ[4][DSACT_MAX_CONV + 1];   // activations 1..nconv
  CnnHeadBuf hb[14];   // 0,1 pi mean/ls; 2,3 pi'; 4..7 Q1,Q2 (s,a) mean/ls; 8..11 Q1',Q2'; 12,13 mean head of Q1,Q2 on (s,a~)
  int64_t logitsP, logitsT, dlogits, new_act, act2, logp_new, logp2, eps1, eps2, z3, z4, outQ[6], dOut[6], dAct[2];
  int64_t dfeat[3], dfa[2];   // dL/dfeature of pi, Q1, Q2; dL/d(feature|act) scratch of the actor path
  int64_t ga, gb;             // conv-backward ping-pong buffers (largest activation)
  int64_t r_obs, r_obs2, r_act, r_rew, r_done, r_logp, r_idx;   // gathered replay minibatch
  dsact_replay rb;
  dsact_replay_u8 rb8;     // the 8-bit image ring, when rb_u8
  bool rb_bound = false, rb_u8 = false;
  int64_t rb_capacity() const { return rb_u8 ? rb8.capacity : rb.capacity; }
  int64_t dev_rb_size = -1;
  int64_t total;
  float* Wp() const { return reinterpret_cast<float*>(buf.workspace); }
  void layout() {
    const int64_t B = cfg.max_batch, A = cfg.act_dim;
    int64_t off = 0;
    auto take = [&](int64_t n) { int64_t o = off; off += round64(n); return o; };
    auto conv_acts = [&](const CnnGeom& g, int64_t* a) { a[0] = -1; for (int j = 1; j <= g.nconv; ++j) a[j] = take(B * g.act_elems(j)); };
    conv_acts(pi, convP); conv_acts(pi, convT);
    for (int k = 0; k < 4; ++k) conv_acts(q, convQ[k]);
    for (int p = 0; p < 14; ++p) {
      const Net& net = p < 4 ? pi.head : q.head;
      for (int j = 0; j < net.L; ++j) { hb[p].z[j] = take(B * net.s[j + 1]); hb[p].h[j] = take(B * net.s[j + 1]); hb[p].dz[j] = take(B * net.s[j + 1]); }
    }
    logitsP = take(B * 2 * A); logitsT = take(B * 2 * A); dlogits = take(B * 2 * A);
    new_act = take(B * A); act2 = take(B * A); logp_new = take(B); logp2 = take(B);
    eps1 = take(B * A); eps2 = take(B * A); z3 = take(B); z4 = take(B);
    for (int p = 0; p < 6; ++p) { outQ[p] = take(B * 2); dOut[p] = take(B * 2); }
    dAct[0] = take(B * A); dAct[1] = take(B * A);
    dfeat[0] = take(B * pi.F); dfeat[1] = take(B * q.F); dfeat[2] = take(B * q.F);
    dfa[0] = take(B * (q.F + A)); dfa[1] = take(B * (q.F + A));
    int64_t big = 0;
    for (int j = 1; j <= q.nconv; ++j) big = big > q.act_elems(j) ? big : q.act_elems(j);
    for (int j = 1; j <= pi.nconv; ++j) big = big > pi.act_elems(j) ? big : pi.act_elems(j);
    ga = take(B * big); gb = take(B * big);
    const int64_t O = (int64_t)cfg.channels * cfg.height * cfg.width;
    r_obs = take(B * O); r_obs2 = take(B * O); r_act = take(B * A); r_rew = take(B); r_done = take(B); r_logp = take(B); r_idx = take(2 * B);
    total = off;
  }
};

// critics: two heads of one output (networks/cnn.py) or one head of two (networks/mlp.py:113-127); policy: mean and
// log_std heads (networks/cnn.py, mlp.py std_type "mlp_separated") or a mean head + learnable row (std_type "parameter")
static void cnn_build_nets(dsact_cnn_handle* h) {
  const dsact_cnn_config& c = h->cfg;
  const bool q1 = c.q_heads == 1, row = c.pi_std == 1, shared = c.pi_std == 2;
  h->q.build(c, c.act_dim, q1 ? 2 : 1, q1 ? 1 : 2, false);
  h->pi.build(c, 0, shared ? 2 * c.act_dim : c.act_dim, (row || shared) ? 1 : 2, row);
}

static int cnn_validate(const dsact_cnn_config* c) {
  if (!c) return fail(DSACT_EINVAL, "null config");
  if (c->abi_version != DSACT_ABI_VERSION) return fail(DSACT_EINVAL, "abi_version %d != %d", c->abi_version, DSACT_ABI_VERSION);
  if (c->channels < 1 || c->height < 1 || c->width < 1 || c->act_dim < 1) return fail(DSACT_EINVAL, "bad observation / action shape");
  if (c->n_conv < 0 || c->n_conv > DSACT_MAX_CONV) return fail(DSACT_EINVAL, "0..%d conv layers supported", DSACT_MAX_CONV);
  if (c->q_heads != 1 && c->q_heads != 2) return fail(DSACT_EINVAL, "q_heads must be 1 (one head, two outputs) or 2 (mean and std heads)");
  if (c->pi_std < 0 || c->pi_std > 2) return fail(DSACT_EINVAL, "pi_std must be 0 (log_std head), 1 (learnable row) or 2 (one head, 2*act_dim outputs)");
  if (c->algo != 0 && c->algo != 1) return fail(DSACT_EINVAL, "algo must be 0 (DSAC_V2 / DSAC-T) or 1 (DSAC_V1)");
  if (c->algo == 1 && !(c->td_bound > 0.0)) return fail(DSACT_EINVAL, "DSAC_V1 needs TD_bound > 0");
  if (c->act_dist != 0 && c->act_dist != 1) return fail(DSACT_EINVAL, "act_dist must be 0 (TanhGaussDistribution) or 1 (GaussDistribution)");
  for (int j = 0; j < c->n_conv; ++j)
    if (c->conv_kernel[j] < 1 || (c->conv_kernel[j] > 4 && c->conv_kernel[j] != 8) || c->conv_stride[j] < 1 || c->conv_channels[j] < 1)
      return fail(DSACT_EINVAL, "conv layer %d: kernel sizes 1..4 and 8 are implemented (the reference's type_1 / type_2 encoders)", j);
  if (c->n_hidden < 1 || c->n_hidden > DSACT_MAX_HIDDEN) return fail(DSACT_EINVAL, "1..%d hidden layers per head", DSACT_MAX_HIDDEN);
  if (c->act_hidden < 0 || c->act_hidden > DSACT_ACT_SELU) return fail(DSACT_EINVAL, "unknown activation");
  if (c->max_batch < 1 || c->delay_update < 1) return fail(DSACT_EINVAL, "bad max_batch / delay_update");
  CnnGeom g;
  if (!g.build(*c, 0, 1, 2, false)) return fail(DSACT_EINVAL, "the conv stack consumes the whole image");
  return DSACT_OK;
}

// ---- head MLPs through the grouped fp32 GEMM -------------------------------------------------------------------------
struct CnnHeadFwd {
  const float* base;     // parameters of this head
  const float* in0; int k0;
  const float* in1; int k1;     // second input segment (the action) or null
  CnnHeadBuf* hbuf;
  bool keep_z;
  float* out; int out_ld;       // head output column(s) inside a packed array
};
static void cnn_heads_forward(dsact_cnn_handle* h, const Net& net, std::vector<CnnHeadFwd>& P, int B, Ctx& c) {
  float* W = h->Wp();
  for (int j = 0; j <= net.L; ++j) {
    size_t i0 = 0;
    while (i0 < P.size()) {
      GemmGroup G;
      G.n = 0;
      for (; i0 < P.size() && G.n < MAXG; ++i0) {
        const CnnHeadFwd& f = P[i0];
        GemmProb p = prob_zero();
        const int in_dim = net.s[j];
        if (j == 0) {
          p.A[0] = f.in0; p.lda[0] = f.k0; p.K[0] = f.k0; p.B[0] = f.base + net.w[0]; p.ldb[0] = in_dim;
          if (f.k1 > 0) { p.A[1] = f.in1; p.lda[1] = f.k1; p.K[1] = f.k1; p.B[1] = f.base + net.w[0] + f.k0; p.ldb[1] = in_dim; }
        } else {
          p.A[0] = W + f.hbuf->h[j - 1]; p.lda[0] = in_dim; p.K[0] = in_dim; p.B[0] = f.base + net.w[j]; p.ldb[0] = in_dim;
        }
        p.M = B; p.N = net.s[j + 1]; p.bias = f.base + net.b[j]; p.act = h->cfg.act_hidden;
        if (j == net.L) { p.C = f.out; p.ldc = f.out_ld; p.epi = EPI_STORE; }
        else { p.C = W + f.hbuf->h[j]; p.ldc = net.s[j + 1]; p.epi = EPI_BIAS_ACT; p.Zout = f.keep_z ? W + f.hbuf->z[j] : nullptr; }
        G.p[G.n++] = p;
      }
      launch_simt(h->num_sms, G, V_FWD, c);
      c.done();
    }
  }
  c.check();
}

struct CnnHeadBwd {
  const float* base;     // parameters of this head
  float* gbase;          // its gradients, or null (actor path through a critic: input gradient only)
  const float* in0; int k0; const float* in1; int k1;   // layer-0 inputs (for the weight gradient)
  CnnHeadBuf* hbuf;
  const float* dout; int dout_ld;   // dL/d(head output) inside a packed array
  float* din;            // [B, k0 + k1] dL/d(layer-0 input), accumulated (+=), or null
};
static void cnn_heads_backward(dsact_cnn_handle* h, const Net& net, std::vector<CnnHeadBwd>& P, int B, Ctx& c) {
  float* W = h->Wp();
  for (int j = net.L; j >= 0; --j) {
    GemmGroup gw, gd;
    gw.n = gd.n = 0;
    auto flush = [&](GemmGroup& G, int variant) { if (G.n) { launch_simt(h->num_sms, G, variant, c); c.done(); G.n = 0; } };
    for (const CnnHeadBwd& f : P) {
      const float* dY = j == net.L ? f.dout : W + f.hbuf->dz[j];
      const int ldy = j == net.L ? f.dout_ld : net.s[j + 1];
      if (f.gbase) {   // dW_j += dY^T X
        auto wgrad = [&](const float* X, int ldx, int col0, int ncols) {
          GemmProb p = prob_zero();
          p.A[0] = dY; p.lda[0] = ldy; p.K[0] = B; p.B[0] = X; p.ldb[0] = ldx;
          p.M = net.s[j + 1]; p.N = ncols; p.C = f.gbase + net.w[j] + col0; p.ldc = net.s[j]; p.epi = EPI_ATOMIC;
          if (gw.n == MAXG) flush(gw, V_WGRAD);
          gw.p[gw.n++] = p;
        };
        if (j == 0) { wgrad(f.in0, f.k0, 0, f.k0); if (f.k1 > 0) wgrad(f.in1, f.k1, f.k0, f.k1); }
        else wgrad(W + f.hbuf->h[j - 1], net.s[j], 0, net.s[j]);
      }
      GemmProb p = prob_zero();   // dX = dY W_j (.) act'(z_{j-1})
      p.A[0] = dY; p.lda[0] = ldy; p.K[0] = net.s[j + 1]; p.B[0] = f.base + net.w[j]; p.ldb[0] = net.s[j];
      p.M = B; p.N = net.s[j];
      if (j >= 1) {
        p.C = W + f.hbuf->dz[j - 1]; p.ldc = net.s[j];
        p.epi = EPI_DACT; p.Zin = W + f.hbuf->z[j - 1]; p.ldz = net.s[j]; p.act = h->cfg.act_hidden;
        p.colsum = f.gbase ? f.gbase + net.b[j - 1] : nullptr;
      } else {
        if (!f.din) continue;
        p.C = f.din; p.ldc = net.s[0]; p.epi = EPI_ATOMIC;   // several heads add into the same input gradient
      }
      if (gd.n == MAXG) flush(gd, V_DGRAD);
      gd.p[gd.n++] = p;
    }
    flush(gw, V_WGRAD);
    flush(gd, V_DGRAD);
  }
  c.check();
}

template <int R>
static void launch_conv_fwd8(const ConvShape& s, long long rows, size_t smem, Ctx& c, const float* x, const float* w, const float* b, float* y) {
  const dim3 grid((unsigned)((rows + 128 * R - 1) / (128 * R)), s.Cout / 8);
  switch (s.K) {
    case 1: launch_k(conv_fwd8_kernel<1, R>, grid, 128, smem, c, x, w, b, y, s); break;
    case 2: launch_k(conv_fwd8_kernel<2, R>, grid, 128, smem, c, x, w, b, y, s); break;
    case 3: launch_k(conv_fwd8_kernel<3, R>, grid, 128, smem, c, x, w, b, y, s); break;
    case 4: launch_k(conv_fwd8_kernel<4, R>, grid, 128, smem, c, x, w, b, y, s); break;
    default:   // 8x8 window (type_1's first layer): one position per thread (64 taps in registers)
      if constexpr (R == 1) launch_k(conv_fwd8_kernel<8, 1>, grid, 128, smem, c, x, w, b, y, s);
      break;
  }
}

// a layer whose window is its whole input is a linear layer over the flattened [Cin*K*K] sample (its NCHW order)
static bool conv_is_linear(const ConvShape& s) { return s.Hin == s.K && s.Win == s.K; }

static void cnn_conv_forward(dsact_cnn_handle* h, const CnnGeom& g, const float* params, const float* img, const int64_t* acts, int B, Ctx& c) {
  float* W = h->Wp();
  const float* x = img;
  for (int j = 0; j < g.nconv; ++j) {
    const ConvShape s = g.shape(j, B);
    const long long rows = (long long)B * s.Hout * s.Wout;
    const size_t smem8 = sizeof(float) * 8 * s.Cin * s.K * s.K;
    if (conv_is_linear(s)) {
      GemmGroup G; G.n = 0;
      GemmProb p = prob_zero();
      const int kin = s.Cin * s.K * s.K;
      p.A[0] = x; p.lda[0] = kin; p.K[0] = kin; p.B[0] = params + g.cw[j]; p.ldb[0] = kin;
      p.M = B; p.N = s.Cout; p.C = W + acts[j + 1]; p.ldc = s.Cout; p.bias = params + g.cb[j]; p.act = ACT_RELU; p.epi = EPI_BIAS_ACT;
      G.p[G.n++] = p;
      launch_simt(h->num_sms, G, V_FWD, c);
    } else if (s.Cout % 8 == 0 && smem8 <= 48 * 1024) {   // eight output channels per thread, 1 / 2 / 4 positions
      const long long wave = 2LL * h->num_sms * 128;
      const float *w = params + g.cw[j], *b = params + g.cb[j];
      if (s.K > 4) launch_conv_fwd8<1>(s, rows, smem8, c, x, w, b, W + acts[j + 1]);
      else if (rows >= 4 * wave) launch_conv_fwd8<4>(s, rows, smem8, c, x, w, b, W + acts[j + 1]);
      else if (rows >= 2 * wave) launch_conv_fwd8<2>(s, rows, smem8, c, x, w, b, W + acts[j + 1]);
      else launch_conv_fwd8<1>(s, rows, smem8, c, x, w, b, W + acts[j + 1]);
    } else {
      dim3 grid((unsigned)((rows + 127) / 128), s.Cout);
      launch_k(conv_fwd_kernel, grid, 128, sizeof(float) * s.Cin * s.K * s.K, c, x, params + g.cw[j], params + g.cb[j], W + acts[j + 1], s);
    }
    c.done();
    x = W + acts[j + 1];
  }
  c.check();
}

template <int COB>
static void launch_conv_wgrad(const ConvShape& s, int slabs, Ctx& c, const float* dy, const float* x, float* dw, float* db) {
  const dim3 grid(s.Cin, s.Cout / COB, slabs);
  switch (s.K) {
    case 1: launch_k(conv_wgrad_kernel<1, COB>, grid, 256, 0, c, dy, x, dw, db, s); break;
    case 2: launch_k(conv_wgrad_kernel<2, COB>, grid, 256, 0, c, dy, x, dw, db, s); break;
    case 3: launch_k(conv_wgrad_kernel<3, COB>, grid, 256, 0, c, dy, x, dw, db, s); break;
    case 4: if constexpr (COB <= 4) launch_k(conv_wgrad_kernel<4, COB>, grid, 256, 0, c, dy, x, dw, db, s); break;
    default: if constexpr (COB == 1) launch_k(conv_wgrad_kernel<8, 1>, grid, 256, 0, c, dy, x, dw, db, s); break;   // 64 taps x 1 channel
  }
}

// backward through one encoder: `gtop` = dL/d(feature) [B, F] (consumed); gparams was cleared by begin_step_kernel
static void cnn_conv_backward(dsact_cnn_handle* h, const CnnGeom& g, const float* params, float* gparams, const float* img,
                              const int64_t* acts, float* gtop, int B, Ctx& c) {
  float* W = h->Wp();
  float* gcur = gtop;
  float* bufs[2] = {W + h->ga, W + h->gb};
  int flip = 0;
  {   // dz of the top layer = g (.) [feature > 0]; the layers below are masked by the dgrad kernel that produces them
    const long long n_out = (long long)B * g.act_elems(g.nconv);
    int blocks = (int)((n_out + 255) / 256); if (blocks > 8 * h->num_sms) blocks = 8 * h->num_sms;
    launch_k(relu_mask_kernel, blocks, 256, 0, c, gcur, (const float*)(W + acts[g.nconv]), n_out); c.done();
  }
  for (int j = g.nconv - 1; j >= 0; --j) {
    const ConvShape s = g.shape(j, B);
    const float* x = j == 0 ? img : W + acts[j];
    const long long rows = (long long)B * s.Hout * s.Wout;
    if (conv_is_linear(s)) {   // dW = dz^T x through the GEMM
      GemmGroup gw; gw.n = 0;
      GemmProb p = prob_zero();
      const int kin = s.Cin * s.K * s.K;
      p.A[0] = gcur; p.lda[0] = s.Cout; p.K[0] = B; p.B[0] = x; p.ldb[0] = kin;
      p.M = s.Cout; p.N = kin; p.C = gparams + g.cw[j]; p.ldc = kin; p.epi = EPI_ATOMIC;
      gw.p[gw.n++] = p;
      launch_simt(h->num_sms, gw, V_WGRAD, c); c.done();
      launch_k(colsum_rows_kernel, (s.Cout + 31) / 32, dim3(32, 8), 0, c, (const float*)gcur, B, s.Cout, gparams + g.cb[j]); c.done();
    } else {
      // slabs: >= 32 rows per thread, enough blocks for ~4 per SM
      const int cob = s.K > 4 ? 1 : (s.Cout % 8 == 0 && s.K <= 3) ? 8 : s.Cout % 4 == 0 ? 4 : 1;   // K*K*cob accumulators per thread
      const int base = s.Cin * (s.Cout / cob);
      long long slabs = (4LL * h->num_sms + base - 1) / base;
      const long long cap = (rows + 256 * 32 - 1) / (256 * 32);
      if (slabs > cap) slabs = cap;
      if (slabs < 1) slabs = 1;
      if (cob == 8) launch_conv_wgrad<8>(s, (int)slabs, c, gcur, x, gparams + g.cw[j], gparams + g.cb[j]);
      else if (cob == 4) launch_conv_wgrad<4>(s, (int)slabs, c, gcur, x, gparams + g.cw[j], gparams + g.cb[j]);
      else launch_conv_wgrad<1>(s, (int)slabs, c, gcur, x, gparams + g.cw[j], gparams + g.cb[j]);
      c.done();
    }
    if (j > 0) {
      float* gnext = bufs[flip]; flip ^= 1;
      const long long rin = (long long)B * s.Hin * s.Win;
      const size_t smem8 = sizeof(float) * 8 * s.Cout * s.K * s.K;
      if (conv_is_linear(s)) {   // dx = dz W (.) [x > 0]
        GemmGroup G; G.n = 0;
        GemmProb p = prob_zero();
        const int kin = s.Cin * s.K * s.K;
        p.A[0] = gcur; p.lda[0] = s.Cout; p.K[0] = s.Cout; p.B[0] = params + g.cw[j]; p.ldb[0] = kin;
        p.M = B; p.N = kin; p.C = gnext; p.ldc = kin; p.epi = EPI_DACT; p.Zin = x; p.ldz = kin; p.act = ACT_RELU;
        G.p[G.n++] = p;
        launch_simt(h->num_sms, G, V_DGRAD, c);
      } else if (s.Cin % 8 == 0 && smem8 <= (size_t)CNN_DGRAD_SMEM) {
        dim3 grid((unsigned)((rin + 127) / 128), s.Cin / 8);
        launch_k(conv_dgrad8_kernel, grid, 128, smem8, c, (const float*)gcur, params + g.cw[j], x, gnext, s, 1);
      } else {
        dim3 grid((unsigned)((rin + 127) / 128), s.Cin);
        launch_k(conv_dgrad_kernel, grid, 128, 0, c, (const float*)gcur, params + g.cw[j], x, gnext, s, 1);
      }
      c.done();
      gcur = gnext;
    }
  }
  c.check();
}

// ---- one DSAC-T step in three parts: forwards (phase 1) | losses + backward (phase 2) | Adam + Polyak (apply) ---------
// dsact_cnn_step enqueues all three; the split entry points enqueue one each, so that a data-parallel caller can
// all-reduce the critics' std sums after phase 1 and the gradients + logged sums after phase 2.
struct CnnSpans {   // per-network slices of the flat buffers
  float *Pq[2], *Ppi, *Tq[2], *Tpi, *Gq[2], *Gpi;
  long long n_all;   // 2 * n_q + n_pi + 1
};
static CnnSpans cnn_spans(const dsact_cnn_handle* h) {
  const int64_t nq = h->q.n;
  float *P = h->buf.params, *T = h->buf.targets, *G = h->buf.grads;
  return CnnSpans{{P, P + nq}, P + 2 * nq, {T, T + nq}, T + 2 * nq, {G, G + nq}, G + 2 * nq, 2 * nq + h->pi.n + 1};
}
// the encoders' outputs; without a conv stack (the MLP approximators with separate heads) the feature is the observation
struct CnnFeatures { const float *P, *T, *Q[4]; bool enc; };
static CnnFeatures cnn_features(const dsact_cnn_handle* h, const dsact_batch& bt) {
  float* W = h->Wp();
  const CnnGeom &q = h->q, &pi = h->pi;
  const bool enc = pi.nconv > 0;
  return CnnFeatures{enc ? W + h->convP[pi.nconv] : bt.obs, enc ? W + h->convT[pi.nconv] : bt.obs2,
                     {enc ? W + h->convQ[0][q.nconv] : bt.obs, enc ? W + h->convQ[1][q.nconv] : bt.obs,
                      enc ? W + h->convQ[2][q.nconv] : bt.obs2, enc ? W + h->convQ[3][q.nconv] : bt.obs2},
                     enc};
}
static StepScalars cnn_scalars(const dsact_cnn_handle* h, int64_t global_batch) {
  StepScalars sc;
  sc.tau_b = (float)h->cfg.tau_b; sc.alpha_fixed = (float)h->cfg.alpha_fixed; sc.inv_global_batch = (float)(1.0 / (double)global_batch);
  sc.auto_alpha = h->cfg.auto_alpha; sc.log_alpha = h->buf.params + 2 * h->q.n + h->pi.n;
  return sc;
}

// clears grads / accumulators, draws the noise (noise == null), runs every forward; sample_kernel leaves the local
// critic-std sums in state[ST_STDSUM..+1].  Records the minibatch and noise for phase 2.
static void cnn_enqueue_phase1(dsact_cnn_handle* h, const dsact_batch& bt, const dsact_noise* noise, Ctx& c) {
  const dsact_cnn_config& cf = h->cfg;
  const CnnGeom &q = h->q, &pi = h->pi;
  const int B = bt.batch, A = cf.act_dim;
  float* W = h->Wp();
  const CnnSpans sp = cnn_spans(h);
  {
    int blocks = (int)((sp.n_all / 4 + 255) / 256); if (blocks > 2 * h->num_sms) blocks = 2 * h->num_sms; if (blocks < 1) blocks = 1;
    launch_k(begin_step_kernel, blocks, 256, 0, c, h->buf.state, h->buf.grads, sp.n_all); c.done();
  }
  const float *eps1, *eps2;
  if (noise) { eps1 = noise->eps1; eps2 = noise->eps2; h->pending_z3 = noise->z3; h->pending_z4 = noise->z4; }
  else {
    const int total = (B * A + 1) / 2 * 2 + (B + 1) / 2 * 2;
    int blocks = (total / 2 + 255) / 256; if (blocks < 1) blocks = 1;
    launch_k(noise_kernel, blocks, 256, 0, c, W + h->eps1, W + h->eps2, W + h->z3, W + h->z4, B, A, h->seed, (const float*)h->buf.state); c.done();
    eps1 = W + h->eps1; eps2 = W + h->eps2; h->pending_z3 = W + h->z3; h->pending_z4 = W + h->z4;
  }
  h->pending_eps1 = eps1;

  // ---- encoders: pi(s), pi'(s'), Q_k features of s, Q'_k features of s'
  cnn_conv_forward(h, pi, sp.Ppi, bt.obs, h->convP, B, c);
  cnn_conv_forward(h, pi, sp.Tpi, bt.obs2, h->convT, B, c);
  for (int k = 0; k < 2; ++k) {
    cnn_conv_forward(h, q, sp.Pq[k], bt.obs, h->convQ[k], B, c);
    cnn_conv_forward(h, q, sp.Tq[k], bt.obs2, h->convQ[2 + k], B, c);
  }
  const CnnFeatures f = cnn_features(h, bt);

  // ---- policy heads: logits = (mean | log_std), the layout sample_kernel reads (networks/cnn.py:233-240)
  {
    std::vector<CnnHeadFwd> v;
    for (int hd = 0; hd < pi.nheads; ++hd) {
      v.push_back({sp.Ppi + pi.head_off[hd], f.P, pi.F, nullptr, 0, &h->hb[hd], true, W + h->logitsP + hd * A, 2 * A});
      v.push_back({sp.Tpi + pi.head_off[hd], f.T, pi.F, nullptr, 0, &h->hb[2 + hd], false, W + h->logitsT + hd * A, 2 * A});
    }
    cnn_heads_forward(h, pi.head, v, B, c);
    if (pi.ls_row >= 0) {   // std_type "parameter": log_std columns = the learnable row
      int blocks = (B * A + 255) / 256; if (blocks > 4 * h->num_sms) blocks = 4 * h->num_sms;
      launch_k(bcast_row_kernel, blocks, 256, 0, c, W + h->logitsP, 2 * A, A, (const float*)(sp.Ppi + pi.ls_row), B, A); c.done();
      launch_k(bcast_row_kernel, blocks, 256, 0, c, W + h->logitsT, 2 * A, A, (const float*)(sp.Tpi + pi.ls_row), B, A); c.done();
    }
  }
  // ---- critics on (s, a): out = (mean, raw std) packed [B,2] (networks/cnn.py:454-461; softplus is applied by the loss kernels)
  {
    std::vector<CnnHeadFwd> v;
    for (int k = 0; k < 2; ++k)
      for (int hd = 0; hd < q.nheads; ++hd)
        v.push_back({sp.Pq[k] + q.head_off[hd], f.Q[k], q.F, bt.act, A, &h->hb[4 + 2 * k + hd], true, W + h->outQ[k] + hd, 2});
    cnn_heads_forward(h, q.head, v, B, c);
  }
  {
    SampleArgs a;
    a.logits[0] = W + h->logitsP; a.logits[1] = W + h->logitsT;
    a.eps[0] = eps1; a.eps[1] = eps2;
    a.act[0] = W + h->new_act; a.act[1] = W + h->act2;
    a.logp[0] = W + h->logp_new; a.logp[1] = W + h->logp2;
    a.hi = h->buf.act_high; a.lo = h->buf.act_low; a.state = h->buf.state;
    a.B = B; a.A = A; a.min_log_std = (float)cf.min_log_std; a.max_log_std = (float)cf.max_log_std; a.gauss = cf.act_dist;
    a.img[0] = ImgOut{nullptr, 0, 1, 0}; a.img[1] = ImgOut{nullptr, 0, 1, 0};
    a.out_q[0] = W + h->outQ[0]; a.out_q[1] = W + h->outQ[1];
    a.advance_rng = noise ? 0 : 1;
    int blocks = (B + 7) / 8; if (blocks > 4 * h->num_sms) blocks = 4 * h->num_sms;
    launch_k(sample_kernel, dim3(blocks, 2), 256, 0, c, a); c.done();
  }
  // ---- targets on (s', a') and the mean heads of the critics on (s, a~)
  {
    std::vector<CnnHeadFwd> v;
    for (int k = 0; k < 2; ++k)
      for (int hd = 0; hd < q.nheads; ++hd)
        v.push_back({sp.Tq[k] + q.head_off[hd], f.Q[2 + k], q.F, W + h->act2, A, &h->hb[8 + 2 * k + hd], false, W + h->outQ[2 + k] + hd, 2});
    for (int k = 0; k < 2; ++k)
      v.push_back({sp.Pq[k] + q.head_off[0], f.Q[k], q.F, W + h->new_act, A, &h->hb[12 + k], true, W + h->outQ[4 + k], 2});
    cnn_heads_forward(h, q.head, v, B, c);
  }
  h->pending = bt;
  h->pending_batch = B;
}

// losses over `global_batch` rows (the local shard is h->pending), every backward pass, and the phase-2 tail: the
// log_alpha gradient of the shard, the commit of the mean_std EMA and the temperature, the Adam scalars of the step
static int cnn_enqueue_phase2(dsact_cnn_handle* h, int64_t global_batch, Ctx& c) {
  const dsact_cnn_config& cf = h->cfg;
  const CnnGeom &q = h->q, &pi = h->pi;
  const dsact_batch& bt = h->pending;
  const int B = bt.batch, A = cf.act_dim;
  float* W = h->Wp();
  const CnnSpans sp = cnn_spans(h);
  const CnnFeatures f = cnn_features(h, bt);
  const float* eps1 = h->pending_eps1;

  // ---- losses and head-output gradients
  const StepScalars sc = cnn_scalars(h, global_batch);
  {
    LossArgs a;
    a.sc = sc;
    a.rew = bt.rew; a.done = bt.done; a.z3 = h->pending_z3; a.z4 = h->pending_z4;
    a.logp2 = W + h->logp2; a.logp_new = W + h->logp_new;
    for (int k = 0; k < 2; ++k) {
      a.out_q[k] = W + h->outQ[k]; a.out_qt[k] = W + h->outQ[2 + k]; a.out_qa[k] = W + h->outQ[4 + k];
      a.d_out_q[k] = W + h->dOut[k]; a.d_out_qa[k] = W + h->dOut[4 + k];
      a.gbias_q[k] = sp.Gq[k] + q.head_off[0] + q.head.b[q.head.L];          // output bias of the mean head
      a.gbias_q_raw[k] = q.nheads == 2 ? sp.Gq[k] + q.head_off[1] + q.head.b[q.head.L] : nullptr;   // ... of the std head (one head: the next element)
      a.img_q[k] = ImgOut{nullptr, 0, 1, 0}; a.img_qa[k] = ImgOut{nullptr, 0, 1, 0};
    }
    a.state = h->buf.state; a.B = B; a.gamma = (float)cf.gamma; a.inv_global_batch = sc.inv_global_batch;
    int blocks = (B + 63) / 64; if (blocks > 4 * h->num_sms) blocks = 4 * h->num_sms;
    launch_k(loss_kernel, blocks, 64, 0, c, a); c.done();
  }
  auto zero = [&](float* p, long long n) {
    int blocks = (int)((n + 255) / 256); if (blocks > 4 * h->num_sms) blocks = 4 * h->num_sms; if (blocks < 1) blocks = 1;
    launch_k(zero_kernel, blocks, 256, 0, c, p, n); c.done();
  };
  zero(W + h->dfeat[0], (long long)B * pi.F);
  zero(W + h->dfeat[1], (long long)B * q.F);
  zero(W + h->dfeat[2], (long long)B * q.F);
  zero(W + h->dfa[0], (long long)B * (q.F + A));
  zero(W + h->dfa[1], (long long)B * (q.F + A));
  // ---- critic backward through both heads (feature gradient accumulated over the heads), actor path through the mean head
  {
    std::vector<CnnHeadBwd> v;
    for (int k = 0; k < 2; ++k)
      for (int hd = 0; hd < q.nheads; ++hd)   // d(feature|act): only the feature part is used (replayed actions carry no gradient)
        v.push_back({sp.Pq[k] + q.head_off[hd], sp.Gq[k] + q.head_off[hd], f.Q[k], q.F, bt.act, A, &h->hb[4 + 2 * k + hd],
                     W + h->dOut[k] + hd, 2, nullptr});
    for (int k = 0; k < 2; ++k)
      v.push_back({sp.Pq[k] + q.head_off[0], nullptr, f.Q[k], q.F, W + h->new_act, A, &h->hb[12 + k], W + h->dOut[4 + k], 2, W + h->dfa[k]});
    cnn_heads_backward(h, q.head, v, B, c);
  }
  // feature gradients of the critics: the layer-0 input gradient of both heads, feature columns only.  The generic
  // backward above skipped it for the critic passes (din = null): do it here with the feature-width problem
  for (int k = 0; k < 2 && f.enc; ++k) {
    GemmGroup gd;
    gd.n = 0;
    for (int hd = 0; hd < q.nheads; ++hd) {
      GemmProb p = prob_zero();
      const Net& net = q.head;
      p.A[0] = W + h->hb[4 + 2 * k + hd].dz[0]; p.lda[0] = net.s[1]; p.K[0] = net.s[1];
      p.B[0] = sp.Pq[k] + q.head_off[hd] + net.w[0]; p.ldb[0] = net.s[0];
      p.M = B; p.N = q.F; p.C = W + h->dfeat[1 + k]; p.ldc = q.F; p.epi = EPI_ATOMIC;
      gd.p[gd.n++] = p;
    }
    launch_simt(h->num_sms, gd, V_DGRAD, c); c.done();
  }
  // dL/da~ through critic k = the action columns of dfa[k]: compact them for policy_grad_kernel
  for (int k = 0; k < 2; ++k) {
    CUDA_TRY(cudaMemcpy2DAsync(W + h->dAct[k], sizeof(float) * A, W + h->dfa[k] + q.F, sizeof(float) * (q.F + A), sizeof(float) * A, B,
                               cudaMemcpyDeviceToDevice, c.s));
  }
  {
    PolicyGradArgs a;
    a.logits = W + h->logitsP; a.eps = eps1; a.d_act1 = W + h->dAct[0]; a.d_act2 = W + h->dAct[1];
    a.hi = h->buf.act_high; a.lo = h->buf.act_low;
    a.d_logits = W + h->dlogits; a.state = h->buf.state;
    a.gbias = sp.Gpi + pi.head_off[0] + pi.head.b[pi.head.L];        // output bias of the mean head [A]
    a.gbias_ls = pi.ls_row >= 0 ? sp.Gpi + pi.ls_row : (pi.nheads == 2 ? sp.Gpi + pi.head_off[1] + pi.head.b[pi.head.L] : nullptr);   // log_std head / row [A]
    a.B = B; a.A = A; a.min_log_std = (float)cf.min_log_std; a.max_log_std = (float)cf.max_log_std; a.gauss = cf.act_dist;
    a.inv_global_batch = sc.inv_global_batch;
    a.img = ImgOut{nullptr, 0, 1, 0};
    a.sc = sc;
    int blocks = (B + 7) / 8; if (blocks > 8 * h->num_sms) blocks = 8 * h->num_sms; if (blocks < 1) blocks = 1;
    launch_k(policy_grad_kernel, blocks, 256, sizeof(float) * 2 * A, c, a); c.done();
  }
  {
    std::vector<CnnHeadBwd> v;
    for (int hd = 0; hd < pi.nheads; ++hd)
      v.push_back({sp.Ppi + pi.head_off[hd], sp.Gpi + pi.head_off[hd], f.P, pi.F, nullptr, 0, &h->hb[hd], W + h->dlogits + hd * A, 2 * A,
                   f.enc ? W + h->dfeat[0] : nullptr});
    cnn_heads_backward(h, pi.head, v, B, c);
  }
  // ---- encoders backward
  if (f.enc) {
    cnn_conv_backward(h, pi, sp.Ppi, sp.Gpi, bt.obs, h->convP, W + h->dfeat[0], B, c);
    for (int k = 0; k < 2; ++k) cnn_conv_backward(h, q, sp.Pq[k], sp.Gq[k], bt.obs, h->convQ[k], W + h->dfeat[1 + k], B, c);
  }

  // ---- end of backward bookkeeping (log_alpha gradient over the local rows, EMA / temperature commit, Adam scalars)
  const AdamHyper hy{cf.lr_q, cf.lr_pi, cf.lr_alpha, cf.adam_beta1, cf.adam_beta2};
  launch_k(phase2_tail_kernel, 1, 32, 0, c, sp.Gpi + pi.n, h->buf.state, sc, -(float)cf.act_dim, B, hy, 1); c.done();
  h->pending_batch = 0;
  return DSACT_OK;
}

// Adam on the three spans + log_alpha, delayed Polyak, step counters.  `scalars_ready` = 1: the phase-2 tail enqueued
// just before (same counters) wrote the step's Adam scalars; 0: form them here (after a separate compute_grads, or when
// `grads` was written from outside).
static void cnn_enqueue_apply(dsact_cnn_handle* h, int scalars_ready, Ctx& c) {
  const dsact_cnn_config& cf = h->cfg;
  const CnnSpans sp = cnn_spans(h);
  ApplyArgs a;
  memset(&a, 0, sizeof(a));
  a.params = h->buf.params; a.targets = h->buf.targets; a.grads = h->buf.grads; a.m = h->buf.adam_m; a.v = h->buf.adam_v;
  a.state = h->buf.state;
  a.n_q2 = 2 * h->q.n; a.n_all = sp.n_all;
  a.delay_update = cf.delay_update; a.auto_alpha = cf.auto_alpha;
  a.hy = AdamHyper{cf.lr_q, cf.lr_pi, cf.lr_alpha, cf.adam_beta1, cf.adam_beta2}; a.scalars_ready = scalars_ready;
  a.eps = (float)cf.adam_eps; a.tau = (float)cf.tau;
  a.omb1 = (float)(1.0 - cf.adam_beta1); a.b2f = (float)cf.adam_beta2; a.omb2 = (float)(1.0 - cf.adam_beta2);
  a.g_lo = 0; a.g_hi = (sp.n_all + 3) / 4; a.finish = 1;
  int blocks = (int)(((sp.n_all + 3) / 4 + 255) / 256); if (blocks > 8 * h->num_sms) blocks = 8 * h->num_sms;
  launch_k(apply_kernel<0>, blocks, 256, 0, c, a); c.done();
}

static int cnn_check_batch(const dsact_cnn_handle* h, const dsact_batch* batch) {
  if (!h || !h->bound) return fail(DSACT_ESTATE, "dsact_cnn_bind has not been called");
  if (!batch || !batch->obs || !batch->act || !batch->rew || !batch->obs2 || !batch->done) return fail(DSACT_EINVAL, "null batch pointer");
  if (batch->batch < 1 || batch->batch > h->cfg.max_batch) return fail(DSACT_EINVAL, "batch %d outside [1, max_batch=%d]", batch->batch, h->cfg.max_batch);
  return DSACT_OK;
}
static int cnn_split_supported(const dsact_cnn_handle* h, const char* fn) {
  if (h && h->cfg.algo == 1) return fail(DSACT_EINVAL, "%s: DSAC_V1 handles (algo = 1) have dsact_cnn_step only", fn);
  return DSACT_OK;
}
static int cnn_sync_iteration(dsact_cnn_handle* h, int64_t iteration, cudaStream_t s) {
  if (iteration < 0 || iteration > 0x7fffffff) return fail(DSACT_EINVAL, "iteration out of range");
  if (h->dev_iter != iteration) { set_iter_kernel<<<1, 32, 0, s>>>(h->buf.state, (int)iteration); CUDA_TRY(cudaGetLastError()); }
  return DSACT_OK;
}
static int cnn_finish(dsact_cnn_handle* h, const Ctx& c) {
  if (c.err != cudaSuccess) return fail(DSACT_ECUDA, "kernel launch failed: %s", cudaGetErrorString(c.err));
  h->launches += c.launches;
  return DSACT_OK;
}

// rows (ptr + i) % capacity of every column: `cols` = (destination, source, bytes per row)
struct RingCol { void* dst; const void* src; int64_t w; };
static int cnn_ring_copy(const RingCol (&cols)[6], int64_t capacity, int64_t n, int64_t ptr, cudaStream_t s) {
  const int64_t first = (ptr + n <= capacity) ? n : capacity - ptr;
  for (const RingCol& c : cols) {
    char* dst = static_cast<char*>(c.dst);
    const char* src = static_cast<const char*>(c.src);
    CUDA_TRY(cudaMemcpyAsync(dst + ptr * c.w, src, first * c.w, cudaMemcpyDefault, s));
    if (first < n) CUDA_TRY(cudaMemcpyAsync(dst, src + first * c.w, (n - first) * c.w, cudaMemcpyDefault, s));
  }
  return DSACT_OK;
}

#include "v1_step.cuh"

extern "C" {

int dsact_cnn_query_layout(const dsact_cnn_config* cfg, dsact_layout* out) {
  int rc = cnn_validate(cfg);
  if (rc) return rc;
  if (!out) return fail(DSACT_EINVAL, "null out");
  dsact_cnn_handle h;
  h.cfg = *cfg;
  cnn_build_nets(&h);
  h.layout();
  const int ncrit = cfg->algo == 1 ? 1 : 2;   // DSAC_V1 has one critic
  out->n_q = h.q.n; out->n_pi = h.pi.n;
  out->n_params = ncrit * h.q.n + h.pi.n + 1;
  out->n_targets = ncrit * h.q.n + h.pi.n;
  out->workspace_bytes = h.total * (int64_t)sizeof(float);
  out->state_floats = ST_FLOATS;
  out->max_batch = cfg->max_batch;
  return DSACT_OK;
}

int dsact_cnn_create(const dsact_cnn_config* cfg, int device, dsact_cnn_handle** out) {
  int rc = cnn_validate(cfg);
  if (rc) return rc;
  if (!out) return fail(DSACT_EINVAL, "null out");
  CUDA_TRY(cudaSetDevice(device));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return fail(DSACT_EARCH, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
  CUDA_TRY(cudaFuncSetAttribute(conv_dgrad8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, CNN_DGRAD_SMEM));
  dsact_cnn_handle* h = new dsact_cnn_handle();
  h->cfg = *cfg;
  h->device = device;
  h->num_sms = prop.multiProcessorCount;
  cnn_build_nets(h);
  h->layout();
  *out = h;
  return DSACT_OK;
}

void dsact_cnn_destroy(dsact_cnn_handle* h) { delete h; }

int dsact_cnn_bind(dsact_cnn_handle* h, const dsact_buffers* b) {
  if (!h || !b) return fail(DSACT_EINVAL, "null argument");
  if (!b->params || !b->targets || !b->grads || !b->adam_m || !b->adam_v || !b->act_high || !b->act_low || !b->state || !b->workspace)
    return fail(DSACT_EINVAL, "null buffer pointer");
  h->buf = *b;
  h->bound = true;
  h->dev_iter = -1;
  h->pending_batch = 0;
  return DSACT_OK;
}

int dsact_cnn_set_carry(dsact_cnn_handle* h, float m1, float m2, int64_t tq, int64_t tp, void* stream) {
  if (!h || !h->bound) return fail(DSACT_ESTATE, "not bound");
  CUDA_TRY(cudaSetDevice(h->device));
  set_carry_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(h->buf.state, m1, m2, (int)tq, (int)tp);
  CUDA_TRY(cudaGetLastError());
  return DSACT_OK;
}

int dsact_cnn_seed(dsact_cnn_handle* h, uint64_t seed) {
  if (!h) return fail(DSACT_EINVAL, "null handle");
  h->seed = seed;
  return DSACT_OK;
}

int dsact_cnn_read_stats(dsact_cnn_handle* h, int64_t global_batch, float* host_out, void* stream) {
  if (!h || !h->bound) return fail(DSACT_ESTATE, "not bound");
  if (!host_out || global_batch < 1) return fail(DSACT_EINVAL, "bad argument");
  CUDA_TRY(cudaSetDevice(h->device));
  // DSAC_V1 logs one entry of the logits row per sample (dsac_v1.py:142-143), DSAC-T the mean over all action dimensions
  const double pol = h->cfg.algo == 1 ? (double)global_batch : (double)global_batch * h->cfg.act_dim;
  finalize_stats_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(h->buf.state, (float)(1.0 / (double)global_batch), (float)(1.0 / pol));
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpyAsync(host_out, h->buf.state + ST_STATS, DSACT_NUM_STATS * sizeof(float), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  return DSACT_OK;
}

int dsact_cnn_replay_bind(dsact_cnn_handle* h, const dsact_replay* rb) {
  if (!h || !rb) return fail(DSACT_EINVAL, "null argument");
  if (!rb->obs || !rb->obs2 || !rb->act || !rb->rew || !rb->done || !rb->logp || rb->capacity < 1) return fail(DSACT_EINVAL, "bad replay buffers");
  h->rb = *rb;
  h->rb_bound = true;
  h->rb_u8 = false;
  h->dev_rb_size = -1;
  return DSACT_OK;
}

int dsact_cnn_replay_bind_u8(dsact_cnn_handle* h, const dsact_replay_u8* rb) {
  if (!h || !rb) return fail(DSACT_EINVAL, "null argument");
  if (h->cfg.n_conv == 0)
    return fail(DSACT_EINVAL, "dsact_cnn_replay_bind_u8: the handle has no conv encoder (n_conv = 0); 8-bit rings hold images on "
                              "the 1/255 grid, vector observations stay in the fp32 ring");
  if (!rb->obs || !rb->obs2 || !rb->act || !rb->rew || !rb->done || !rb->logp || rb->capacity < 1) return fail(DSACT_EINVAL, "bad replay buffers");
  h->rb8 = *rb;
  h->rb_bound = true;
  h->rb_u8 = true;
  h->dev_rb_size = -1;
  return DSACT_OK;
}

int dsact_cnn_replay_add_u8(dsact_cnn_handle* h, const uint8_t* obs, const uint8_t* obs2, const float* act, const float* rew,
                            const float* done, const float* logp, int64_t n, int64_t ptr, void* stream) {
  if (!h || !h->rb_bound) return fail(DSACT_ESTATE, "replay buffer not bound");
  if (!h->rb_u8) return fail(DSACT_ESTATE, "dsact_cnn_replay_add_u8: the bound ring stores fp32 images; use dsact_cnn_replay_add");
  if (n < 0 || n > h->rb8.capacity || ptr < 0 || ptr >= h->rb8.capacity) return fail(DSACT_EINVAL, "bad n/ptr");
  if (n == 0) return DSACT_OK;
  if (!obs || !obs2 || !act || !rew || !done || !logp) return fail(DSACT_EINVAL, "null staging pointer");
  CUDA_TRY(cudaSetDevice(h->device));
  const int64_t O = (int64_t)h->cfg.channels * h->cfg.height * h->cfg.width, A = h->cfg.act_dim;
  const int64_t f = sizeof(float);
  const RingCol cols[6] = {{h->rb8.obs, obs, O}, {h->rb8.obs2, obs2, O}, {h->rb8.act, act, A * f},
                           {h->rb8.rew, rew, f}, {h->rb8.done, done, f}, {h->rb8.logp, logp, f}};
  return cnn_ring_copy(cols, h->rb8.capacity, n, ptr, (cudaStream_t)stream);
}

int dsact_cnn_replay_add(dsact_cnn_handle* h, const float* obs, const float* obs2, const float* act, const float* rew,
                         const float* done, const float* logp, int64_t n, int64_t ptr, void* stream) {
  if (!h || !h->rb_bound) return fail(DSACT_ESTATE, "replay buffer not bound");
  if (h->rb_u8) return fail(DSACT_ESTATE, "dsact_cnn_replay_add: the bound ring stores 8-bit images; use dsact_cnn_replay_add_u8");
  if (n < 0 || n > h->rb.capacity || ptr < 0 || ptr >= h->rb.capacity) return fail(DSACT_EINVAL, "bad n/ptr");
  if (n == 0) return DSACT_OK;
  if (!obs || !obs2 || !act || !rew || !done || !logp) return fail(DSACT_EINVAL, "null staging pointer");
  CUDA_TRY(cudaSetDevice(h->device));
  const int64_t O = (int64_t)h->cfg.channels * h->cfg.height * h->cfg.width, A = h->cfg.act_dim;
  const int64_t f = sizeof(float);
  const RingCol cols[6] = {{h->rb.obs, obs, O * f}, {h->rb.obs2, obs2, O * f}, {h->rb.act, act, A * f},
                           {h->rb.rew, rew, f}, {h->rb.done, done, f}, {h->rb.logp, logp, f}};
  return cnn_ring_copy(cols, h->rb.capacity, n, ptr, (cudaStream_t)stream);
}

int dsact_cnn_replay_sample(dsact_cnn_handle* h, int32_t batch, int64_t size, const int64_t* idx, dsact_batch* out, void* stream) {
  if (!h || !h->bound || !h->rb_bound) return fail(DSACT_ESTATE, "not bound");
  if (batch < 1 || batch > h->cfg.max_batch) return fail(DSACT_EINVAL, "batch outside [1, max_batch]");
  if (size < 1 || size > h->rb_capacity()) return fail(DSACT_EINVAL, "size %lld outside [1, capacity]", (long long)size);
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  if (h->dev_rb_size != size) { set_rb_size_kernel<<<1, 32, 0, s>>>(h->buf.state, size); CUDA_TRY(cudaGetLastError()); h->dev_rb_size = size; }
  float* W = h->Wp();
  const int O = h->cfg.channels * h->cfg.height * h->cfg.width, A = h->cfg.act_dim;
  Ctx c{s, 0, cudaSuccess};
  c.pdl = false;
  int64_t* draw = idx ? nullptr : reinterpret_cast<int64_t*>(W + h->r_idx);
  int blocks = (batch + 7) / 8; if (blocks > 8 * h->num_sms) blocks = 8 * h->num_sms;
  const ImgOut none{nullptr, 0, 1, 0};
  if (h->rb_u8) {
    const int wpb = GATHER_U8_THREADS / 32;
    int b8 = (batch + wpb - 1) / wpb; if (b8 > 32 * h->num_sms) b8 = 32 * h->num_sms;
    launch_k(gather_u8_kernel, b8, GATHER_U8_THREADS, 0, c, (const uint8_t*)h->rb8.obs, (const uint8_t*)h->rb8.obs2, (const float*)h->rb8.act,
             (const float*)h->rb8.rew, (const float*)h->rb8.done, (const float*)h->rb8.logp, idx, W + h->r_obs, W + h->r_obs2, W + h->r_act,
             W + h->r_rew, W + h->r_done, W + h->r_logp, (int)batch, O, A, draw, (unsigned long long)h->seed, (const float*)h->buf.state);
  } else {
    launch_k(gather_kernel, blocks, 256, 0, c, (const float*)h->rb.obs, (const float*)h->rb.obs2, (const float*)h->rb.act, (const float*)h->rb.rew,
             (const float*)h->rb.done, (const float*)h->rb.logp, idx, W + h->r_obs, W + h->r_obs2, W + h->r_act, W + h->r_rew, W + h->r_done,
             W + h->r_logp, (int)batch, O, A, none, none, none, draw, (unsigned long long)h->seed, (const float*)h->buf.state, 1);
  }
  c.done();
  if (!idx) { launch_k(rng_advance_kernel, 1, 32, 0, c, h->buf.state); c.done(); }
  if (c.err != cudaSuccess) return fail(DSACT_ECUDA, "kernel launch failed: %s", cudaGetErrorString(c.err));
  h->launches += c.launches;
  if (out) {
    out->obs = W + h->r_obs; out->act = W + h->r_act; out->rew = W + h->r_rew; out->obs2 = W + h->r_obs2; out->done = W + h->r_done;
    out->logp = W + h->r_logp; out->batch = batch;
  }
  return DSACT_OK;
}

int dsact_cnn_step(dsact_cnn_handle* h, const dsact_batch* batch, const dsact_noise* noise, int64_t iteration, void* stream) {
  int rc = cnn_check_batch(h, batch);
  if (rc || (rc = check_noise(noise))) return rc;
  if (iteration < 0 || iteration > 0x7fffffff) return fail(DSACT_EINVAL, "iteration out of range");
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  if ((rc = cnn_sync_iteration(h, iteration, s))) return rc;
  if (h->cfg.algo == 1) return cnn_step_v1(h, batch, noise, iteration, s);
  Ctx c{s, 0, cudaSuccess};
  c.pdl = false;
  cnn_enqueue_phase1(h, *batch, noise, c);
  rc = cnn_enqueue_phase2(h, batch->batch, c);
  if (rc) { h->pending_batch = 0; return rc; }
  cnn_enqueue_apply(h, 1, c);
  if ((rc = cnn_finish(h, c))) return rc;
  h->dev_iter = iteration + 1;
  return DSACT_OK;
}

int dsact_cnn_grad_phase1(dsact_cnn_handle* h, const dsact_batch* batch, const dsact_noise* noise, void* stream) {
  int rc = cnn_check_batch(h, batch);
  if (rc || (rc = check_noise(noise)) || (rc = cnn_split_supported(h, "dsact_cnn_grad_phase1"))) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  Ctx c{(cudaStream_t)stream, 0, cudaSuccess};
  c.pdl = false;
  cnn_enqueue_phase1(h, *batch, noise, c);
  if ((rc = cnn_finish(h, c))) h->pending_batch = 0;
  return rc;
}

int dsact_cnn_grad_phase2(dsact_cnn_handle* h, int64_t global_batch, void* stream) {
  if (!h || !h->bound) return fail(DSACT_ESTATE, "dsact_cnn_bind has not been called");
  int rc = cnn_split_supported(h, "dsact_cnn_grad_phase2");
  if (rc) return rc;
  if (h->pending_batch < 1) return fail(DSACT_ESTATE, "dsact_cnn_grad_phase2 without a preceding dsact_cnn_grad_phase1");
  if (global_batch < h->pending_batch || global_batch > 0x7fffffff)
    return fail(DSACT_EINVAL, "global_batch %lld outside [local batch %d, 2^31)", (long long)global_batch, h->pending_batch);
  CUDA_TRY(cudaSetDevice(h->device));
  Ctx c{(cudaStream_t)stream, 0, cudaSuccess};
  c.pdl = false;
  rc = cnn_enqueue_phase2(h, global_batch, c);
  h->pending_batch = 0;
  return rc ? rc : cnn_finish(h, c);
}

int dsact_cnn_compute_grads(dsact_cnn_handle* h, const dsact_batch* batch, const dsact_noise* noise, void* stream) {
  int rc = cnn_check_batch(h, batch);
  if (rc || (rc = check_noise(noise)) || (rc = cnn_split_supported(h, "dsact_cnn_compute_grads"))) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  Ctx c{(cudaStream_t)stream, 0, cudaSuccess};
  c.pdl = false;
  cnn_enqueue_phase1(h, *batch, noise, c);
  rc = cnn_enqueue_phase2(h, batch->batch, c);
  h->pending_batch = 0;
  return rc ? rc : cnn_finish(h, c);
}

int dsact_cnn_apply(dsact_cnn_handle* h, int64_t iteration, void* stream) {
  if (!h || !h->bound) return fail(DSACT_ESTATE, "dsact_cnn_bind has not been called");
  int rc = cnn_split_supported(h, "dsact_cnn_apply");
  if (rc) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  if ((rc = cnn_sync_iteration(h, iteration, s))) return rc;
  Ctx c{s, 0, cudaSuccess};
  c.pdl = false;
  cnn_enqueue_apply(h, 0, c);
  if ((rc = cnn_finish(h, c))) return rc;
  h->dev_iter = iteration + 1;
  return DSACT_OK;
}

}  // extern "C"
