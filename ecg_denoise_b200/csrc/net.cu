// net.cu -- whole-network schedule of RA-LENet (ralenet.forward, model/transformer.py:621-667 and
// raletransformer.py:640-680) and its backward: one host call enqueues every kernel on the stream.
//
//   stem -> [2 blocks @ s0] -> pm1 -> [2 @ s1] -> pm2 -> [2 @ s2] -> pm3 -> [2 @ s3] -> pm4
//        -> [2 @ s4] (+x4) -> [2 @ s4] -> ps4 (+x3) -> [2 @ s3] -> ps3 (+x2) -> [2 @ s2] -> ps2 (+x1)
//        -> [2 @ s1] -> ps1 -> (+stem) head
//
// stage s: C = 8<<s channels, L = L0>>s tokens, H = 2<<s heads; every activation is L*C = 8*L0 floats
// per window.  The workspace is carved deterministically from (B, L0, save, flags) so forward and backward
// agree on where each saved tensor lives.
#include "common.cuh"
#include <algorithm>

namespace {

struct BlockGeom {
  int stage;   // 0..4
  int rw;      // R-wave table index 0..3 or -1
};
// forward order, see rl_net_ptrs
const BlockGeom kBlocks[RL_NBLOCKS] = {{0, 0}, {0, 0}, {1, 1}, {1, 1}, {2, 2},  {2, 2},  {3, 3},  {3, 3},  {4, -1},
                                       {4, -1}, {4, -1}, {4, -1}, {3, 3}, {3, 3}, {2, 2}, {2, 2}, {1, 1}, {1, 1}};
const int kRwWindow[4] = {32, 16, 8, 4};   // model/transformer.py:576-579

struct BlockWs {
  float *xa, *y, *q, *k, *v, *o, *lse, *h;
};
struct Ws {
  float* x0;
  BlockWs blk[RL_NBLOCKS];
  float *pm_out[4], *pm_u[4], *ps_out[4], *ps_u[4];
  // two sets of weight-gradient scratch (alternating per block) and four rotating gradient buffers: the
  // weight-gradient GEMMs run on a side stream up to three kernels behind the data-gradient chain
  float *dqkv[2], *ua[2], *dh[2], *g2[2], *uf[2], *gsum, *grot[4], *gskip[5], *gx0, *gfirst, *partials;
  float *ping, *pong;   // inference only
  // RL_NET_DETERMINISTIC: partial slabs of the attention / feed-forward backward kernels (two sets, alternating per
  // block like dqkv / dh), of the patch kernels, and of the head / stem kernels (reduced on the main stream)
  float *det_attn[2], *det_ffn[2], *det_patch, *det_ends;
  size_t det_attn_n, det_ffn_n, det_patch_n, det_ends_n;
  size_t floats;
};

// Partial-slab floats of one backward kernel (with its weight-gradient GEMMs) of each kind: upper bounds over the
// stages, a function of (B, L0) alone; rl_det_take() checks every slab against them.  Slots: one per CTA of the
// in-CTA gradients (B windows, or ceil(B L / 128) * NSL <= B / 2 + 4 token-tile CTAs at the tcgen05 feed-forward
// stages), one per token slice of the GEMMs (<= min(RL_DET_MAX_SPLIT, ceil(M / 64)) in every GEMM family).
struct DetSizes {
  size_t attn, ffn, patch, ends;
};
DetSizes det_sizes(int B, int L0) {
  const size_t cta = (size_t)B + 4, slack = 4 * RL_DET_MAXRED;
  auto gemm = [](size_t M) { return std::min<size_t>(RL_DET_MAX_SPLIT, (M + 63) / 64); };
  DetSizes d = {0, 0, 0, slack + 56 * (size_t)B};
  for (int s = 0; s < 5; ++s) {
    const size_t C = 8u << s, L = (size_t)L0 >> s, M = (size_t)B * L;
    const size_t wslots = (C <= RL_FW_MAXC) ? cta : gemm(M);
    d.attn = std::max(d.attn, slack + (2 * C + 128) * cta + (4 * C * C + 4 * C) * wslots);   // LN, R-wave table | weights
    d.ffn = std::max(d.ffn, slack + (2 * C + 12 * C) * cta + (8 * C * C + 5 * C) * wslots);  // LN, lew | weights
    for (int mode = 0; mode < 2; ++mode) {                                                  // merge 2C / separate C/2
      const size_t CN = mode == 0 ? 2 * C : C / 2;
      if (CN < 8 || CN > 128) continue;
      d.patch = std::max(d.patch, slack + 2 * CN * cta + CN * CN * gemm(M * C / CN));
    }
  }
  return d;
}

Ws carve(float* base, int B, int L0, int save, int flags) {
  Ws w;
  const size_t N = (size_t)B * 8 * L0;
  size_t off = 0;
  auto take = [&](size_t n) {
    float* p = base ? base + off : nullptr;
    off += (n + 63) & ~(size_t)63;     // keep every buffer 256-byte aligned
    return p;
  };
  w.x0 = take(N);
  for (int j = 0; j < 4; ++j) w.pm_out[j] = take(N);
  w.partials = take((size_t)B * 16);
  if (save) {
    for (int i = 0; i < RL_NBLOCKS; ++i) {
      BlockWs& b = w.blk[i];
      b.xa = take(N); b.y = take(N); b.q = take(N); b.k = take(N); b.v = take(N); b.o = take(N);
      b.lse = take(N / 4); b.h = take(4 * N);
    }
    for (int j = 0; j < 4; ++j) { w.pm_u[j] = take(N); w.ps_out[j] = take(N); w.ps_u[j] = take(N); }
    for (int p = 0; p < 2; ++p) {
      w.dqkv[p] = take(3 * N); w.ua[p] = take(N); w.dh[p] = take(4 * N); w.g2[p] = take(4 * N); w.uf[p] = take(N);
    }
    w.gsum = take(N);
    for (int p = 0; p < 4; ++p) w.grot[p] = take(N);
    w.gskip[0] = nullptr;
    for (int j = 1; j <= 4; ++j) w.gskip[j] = take(N);
    w.gx0 = take(N);
    w.gfirst = take(N);
    w.ping = w.pong = nullptr;
    if (flags & RL_NET_DETERMINISTIC) {
      const DetSizes d = det_sizes(B, L0);
      for (int p = 0; p < 2; ++p) { w.det_attn[p] = take(d.attn); w.det_ffn[p] = take(d.ffn); }
      w.det_patch = take(d.patch);
      w.det_ends = take(d.ends);
      w.det_attn_n = d.attn; w.det_ffn_n = d.ffn; w.det_patch_n = d.patch; w.det_ends_n = d.ends;
    }
  } else {
    w.ping = take(N);
    w.pong = take(N);
  }
  w.floats = off;
  return w;
}

int check_cfg(const rl_net_cfg* cfg, const rl_net_ptrs* P) {
  RL_REQUIRE(cfg && P, RL_ERR_NULL, "net: NULL cfg/params");
  RL_REQUIRE(cfg->B > 0 && (cfg->L0 == 256 || cfg->L0 == 512), RL_ERR_SHAPE, "net: unsupported B=%d L0=%d", cfg->B,
             cfg->L0);
  RL_REQUIRE(!(P->table[0] && cfg->L0 != 256), RL_ERR_SHAPE,
             "net: the R-wave bias tables are defined for 256-sample windows only (model/transformer.py:568-579)");
  RL_REQUIRE((cfg->flags & ~(RL_NET_DETERMINISTIC | RL_NET_TF32)) == 0, RL_ERR_SHAPE, "net: unknown flags 0x%x",
             cfg->flags);
  RL_REQUIRE(cfg->ws && cfg->ws_bytes >= ralenet_net_workspace_bytes_ex(cfg->B, cfg->L0, cfg->save, cfg->flags),
             RL_ERR_NULL, "net: workspace missing or too small (%llu bytes given)", (unsigned long long)cfg->ws_bytes);
  RL_REQUIRE(cfg->running_mean && cfg->running_var && cfg->bn_stats, RL_ERR_NULL, "net: BN buffers missing");
  for (int s = 0; s < 5; ++s) RL_REQUIRE(cfg->pe[s], RL_ERR_NULL, "net: positional table %d missing", s);
  return RL_OK;
}

// Side stream for the weight-gradient GEMMs of the backward pass.  One context per host thread (backward runs on
// autograd threads), created on first use; events carry no timing.  Under stream capture the fork / join below
// becomes parallel branches of the captured graph.
struct SideCtx {
  bool ready = false;
  int dev = -1;
  cudaStream_t side = nullptr;
  cudaEvent_t ev_main[4], ev_side[4];
};
thread_local SideCtx g_side;

int side_ctx(SideCtx** out) {
  int dev = 0;
  cudaGetDevice(&dev);
  if (!g_side.ready || g_side.dev != dev) {
    // RALENET_SIDE_PRIO (A/B switch): priority of the weight-gradient stream (0 = lowest = default; negative = higher).
    // Kernel nodes captured into a CUDA graph inherit the priority of the stream they were captured on.
    const char* pe = getenv("RALENET_SIDE_PRIO");
    cudaError_t e = cudaStreamCreateWithPriority(&g_side.side, cudaStreamNonBlocking, pe ? atoi(pe) : 0);
    for (int i = 0; i < 4 && e == cudaSuccess; ++i) {
      e = cudaEventCreateWithFlags(&g_side.ev_main[i], cudaEventDisableTiming);
      if (e == cudaSuccess) e = cudaEventCreateWithFlags(&g_side.ev_side[i], cudaEventDisableTiming);
    }
    RL_REQUIRE(e == cudaSuccess, RL_ERR_CUDA, "net_bwd: side stream setup failed: %s", cudaGetErrorString(e));
    g_side.ready = true;
    g_side.dev = dev;
  }
  *out = &g_side;
  return RL_OK;
}

void fill_stem(rl_stem_args* sa, const rl_net_cfg* cfg, const rl_net_ptrs* P, const float* x, const Ws& w) {
  sa->B = cfg->B; sa->L = cfg->L0; sa->training = cfg->training; sa->_pad = 0;
  sa->x = x; sa->conv_w = P->stem[0]; sa->conv_b = P->stem[1]; sa->bn_w = P->stem[2]; sa->bn_b = P->stem[3];
  sa->running_mean = cfg->running_mean; sa->running_var = cfg->running_var;
  sa->num_batches_tracked = cfg->num_batches_tracked;
  sa->stats = cfg->bn_stats; sa->partials = w.partials; sa->y = w.x0;
  sa->momentum = 0.1f; sa->eps = 1e-5f;
}

}  // namespace

extern "C" uint64_t ralenet_net_workspace_bytes_ex(int32_t B, int32_t L0, int32_t save, int32_t flags) {
  if (B <= 0 || L0 <= 0) return 0;
  return (uint64_t)carve(nullptr, B, L0, save, flags).floats * sizeof(float);
}

extern "C" uint64_t ralenet_net_workspace_bytes(int32_t B, int32_t L0, int32_t save) {
  return ralenet_net_workspace_bytes_ex(B, L0, save, 0);
}

extern "C" int ralenet_net_fwd_stats(const rl_net_cfg* cfg, const rl_net_ptrs* P, const float* x, void* stream) {
  if (int rc = check_cfg(cfg, P)) return rc;
  RL_REQUIRE(x, RL_ERR_NULL, "net_fwd_stats: x is NULL");
  const Ws w = carve((float*)cfg->ws, cfg->B, cfg->L0, cfg->save, cfg->flags);
  rl_stem_args sa;
  fill_stem(&sa, cfg, P, x, w);
  return ralenet_stem_stats(&sa, stream);
}

extern "C" int ralenet_net_fwd(const rl_net_cfg* cfg, const rl_net_ptrs* P, const float* x, float* out, void* stream) {
  if (int rc = check_cfg(cfg, P)) return rc;
  RL_REQUIRE(x && out, RL_ERR_NULL, "net_fwd: x/out is NULL");
  RL_REQUIRE(!(cfg->flags & RL_NET_TF32) || !cfg->save, RL_ERR_SHAPE,
             "net_fwd: RL_NET_TF32 is an inference precision (save must be 0: no backward may use a TF32 forward)");
  const int B = cfg->B, L0 = cfg->L0, save = cfg->save;
  const int32_t blk_flags = RL_F_PRENORM | RL_F_RESIDUAL | ((cfg->flags & RL_NET_TF32) ? RL_F_TF32 : 0);
  const Ws w = carve((float*)cfg->ws, B, L0, save, cfg->flags);
  int rc;
  {
    rl_stem_args sa;
    fill_stem(&sa, cfg, P, x, w);
    if ((rc = ralenet_stem_apply(&sa, stream))) return rc;
  }
  const float* cur = w.x0;
  int ping = 0;
  auto next_buf = [&]() { ping ^= 1; return ping ? w.ping : w.pong; };
  for (int i = 0; i < RL_NBLOCKS; ++i) {
    const int s = kBlocks[i].stage, rwi = kBlocks[i].rw;
    const int C = 8 << s, L = L0 >> s, H = 2 << s;
    float* const* bp = P->blk[i];
    rl_attn_fwd_args aa = {};
    aa.B = B; aa.L = L; aa.C = C; aa.H = H;
    const bool has_rw = rwi >= 0 && P->table[rwi] != nullptr;
    aa.W = has_rw ? kRwWindow[rwi] : 0;
    aa.c0 = has_rw ? (L - aa.W) / 2 : 0;
    aa.flags = blk_flags;
    aa.x = cur; aa.pe = cfg->pe[s];
    aa.ln_w = bp[RL_BLK_LN1W]; aa.ln_b = bp[RL_BLK_LN1B];
    aa.wq = bp[RL_BLK_WQ]; aa.bq = bp[RL_BLK_BQ]; aa.wkv = bp[RL_BLK_WKV]; aa.bkv = bp[RL_BLK_BKV];
    aa.wp = bp[RL_BLK_WP]; aa.bp = bp[RL_BLK_BP];
    aa.table = has_rw ? P->table[rwi] : nullptr;
    if (save) {
      const BlockWs& b = w.blk[i];
      aa.y = b.xa; aa.q = b.q; aa.k = b.k; aa.v = b.v; aa.o = b.o; aa.lse = b.lse;
    } else {
      aa.y = next_buf();
    }
    rl_ffn_fwd_args fa = {};
    fa.B = B; fa.L = L; fa.C = C; fa.le_mode = cfg->le_mode; fa.flags = blk_flags;
    fa.x = aa.y;
    fa.extra = (i == 9) ? w.pm_out[3] : nullptr;                    // x_mid += x4 (transformer.py:646)
    fa.ln_w = bp[RL_BLK_LN2W]; fa.ln_b = bp[RL_BLK_LN2B];
    fa.w1 = bp[RL_BLK_W1]; fa.b1 = bp[RL_BLK_B1]; fa.w2 = bp[RL_BLK_W2]; fa.b2 = bp[RL_BLK_B2];
    fa.lew = bp[RL_BLK_LEW];
    if (save) { fa.y = w.blk[i].y; fa.h = w.blk[i].h; } else { fa.y = next_buf(); fa.h = nullptr; }
    if ((rc = ralenet_block_fwd(&aa, &fa, stream))) return rc;      // one launch at the narrow stages
    cur = fa.y;

    if (i % 2 == 1) {
      const int layer = i / 2;                                      // 0..8
      if (layer < 4) {                                              // pm1..pm4 (transformer.py:633-642)
        rl_patch_fwd_args pa = {};
        pa.B = B; pa.L = L; pa.C = C; pa.mode = 0;
        pa.x = cur; pa.skip = nullptr;
        pa.w = P->pm[layer][0]; pa.ln_w = P->pm[layer][1]; pa.ln_b = P->pm[layer][2];
        pa.y = w.pm_out[layer];
        pa.u = save ? w.pm_u[layer] : nullptr;
        if ((rc = ralenet_patch_fwd(&pa, stream))) return rc;
        cur = pa.y;
      } else if (layer >= 5) {                                      // ps4..ps1 (transformer.py:649-661)
        const int j = 8 - layer;                                    // layer 5 -> ps4 (index 3) ... 8 -> ps1 (0)
        rl_patch_fwd_args pa = {};
        pa.B = B; pa.L = L; pa.C = C; pa.mode = 1;
        pa.x = cur;
        pa.skip = (j >= 1) ? w.pm_out[j - 1] : nullptr;             // ps4 + x3, ps3 + x2, ps2 + x1, ps1 alone
        pa.w = P->ps[j][0]; pa.ln_w = P->ps[j][1]; pa.ln_b = P->ps[j][2];
        pa.y = save ? w.ps_out[j] : next_buf();
        pa.u = save ? w.ps_u[j] : nullptr;
        if ((rc = ralenet_patch_fwd(&pa, stream))) return rc;
        cur = pa.y;
      }
    }
  }
  rl_head_fwd_args ha = {};
  ha.B = B; ha.L = L0; ha.x = cur; ha.skip = w.x0; ha.w = P->head[0]; ha.b = P->head[1]; ha.out = out;
  return ralenet_head_fwd(&ha, stream);
}

extern "C" int ralenet_net_bwd(const rl_net_cfg* cfg, const rl_net_ptrs* P, const rl_net_ptrs* G, const float* x,
                               const float* dout, void* stream) {
  if (int rc = check_cfg(cfg, P)) return rc;
  RL_REQUIRE(G && x && dout, RL_ERR_NULL, "net_bwd: NULL argument");
  RL_REQUIRE(cfg->save, RL_ERR_SHAPE, "net_bwd: forward was run without save");
  RL_REQUIRE(!(cfg->flags & RL_NET_TF32), RL_ERR_SHAPE, "net_bwd: RL_NET_TF32 is an inference precision");
  const int B = cfg->B, L0 = cfg->L0;
  const Ws w = carve((float*)cfg->ws, B, L0, 1, cfg->flags);
  const bool det = cfg->flags & RL_NET_DETERMINISTIC;
  RlDet dk;   // deterministic mode: partial slabs of the kernel being enqueued (reduced at the end of its fork)
  auto det_on = [&](float* slab, size_t cap) -> RlDet* {
    if (!det) return nullptr;
    dk = RlDet{slab, cap, 0, {}, 0};
    return &dk;
  };
  int rc;
  // input of block i (forward): output of the previous layer piece
  auto block_input = [&](int i) -> const float* {
    if (i % 2 == 1) return w.blk[i - 1].y;
    const int layer = i / 2;
    if (layer == 0) return w.x0;
    if (layer <= 4) return w.pm_out[layer - 1];
    if (layer == 5) return w.blk[9].y;             // x_mid
    return w.ps_out[9 - layer];                    // layer 6 -> ps4 (3), 7 -> ps3 (2), 8 -> ps2 (1)
  };
  {
    rl_head_bwd_args ha = {};
    ha.B = B; ha.L = L0; ha.dout = dout; ha.x = w.ps_out[0]; ha.skip = w.x0; ha.w = P->head[0];
    ha.ds = w.gx0; ha.d_w = G->head[0]; ha.d_b = G->head[1];
    if ((rc = rl_head_bwd(&ha, (cudaStream_t)stream, det_on(w.det_ends, w.det_ends_n)))) return rc;
  }
  const float* g = w.gx0;          // gradient w.r.t. the output of the piece about to be differentiated
  // Main chain: patch / feed-forward / attention data-gradient kernels, numbered n = 0, 1, ...; kernel n writes
  // its data gradient to the rotating buffer grot[n % 4] (unless it has a dedicated destination) and its
  // weight-gradient scratch to set (block & 1).  The weight-gradient GEMMs of kernel n are forked to the side
  // stream; before kernel n starts, the main stream waits for the GEMMs of kernel n - 3 (and, the side stream
  // being in-order, of every earlier one), which are the last readers of everything kernel n overwrites.
  cudaStream_t st_main = (cudaStream_t)stream;
  SideCtx* sc = nullptr;
  const bool use_side = !rl_prof_active();
  if (use_side)
    if ((rc = side_ctx(&sc))) return rc;
  int n = 0;
  int side_idx[4] = {-1, -1, -1, -1};
  int last_side = -1;
  auto before_main = [&]() {
    const int slot = (n + 1) & 3;                 // == (n - 3) mod 4
    if (use_side && n >= 3 && side_idx[slot] == n - 3) cudaStreamWaitEvent(st_main, sc->ev_side[slot], 0);
  };
  auto rot = [&]() { return w.grot[n & 3]; };
  // fork the weight gradients of main kernel n; `launch` enqueues them on the given stream
  auto fork_wgrad = [&](bool has, auto launch) -> int {
    if (!has) return RL_OK;
#ifdef RL_DEBUG_SKIP_WGRAD     // timing experiment only (wrong gradients): what do the side-stream GEMMs cost the main chain?
    return RL_OK;
#endif
    if (!use_side) return launch(st_main);
    const int slot = n & 3;
    cudaEventRecord(sc->ev_main[slot], st_main);
    cudaStreamWaitEvent(sc->side, sc->ev_main[slot], 0);
    if (int r2 = launch(sc->side)) return r2;
    cudaEventRecord(sc->ev_side[slot], sc->side);
    side_idx[slot] = n;
    last_side = slot;
    return RL_OK;
  };
  // the same for a kernel whose parameter gradients went to the partial slabs in *d (deterministic mode): the fork
  // also carries the reduction of every slab, after the GEMMs
  auto fork_grads = [&](bool has, RlDet* d, auto launch) -> int {
    return fork_wgrad(has || (d && d->nred > 0), [&](cudaStream_t q) -> int {
      if (int r2 = launch(q)) return r2;
      return d ? rl_launch_grad_reduce(d, q) : RL_OK;
    });
  };
  for (int i = RL_NBLOCKS - 1; i >= 0; --i) {
    const int s = kBlocks[i].stage, rwi = kBlocks[i].rw;
    const int C = 8 << s, L = L0 >> s, H = 2 << s;
    const int layer = i / 2;
    const int set = i & 1;
    float* const* bp = P->blk[i];
    float* const* bg = G->blk[i];
    const float* g_extra_for_pm = nullptr;
    if (i % 2 == 1) {
      // undo the patch op that followed this layer
      if (layer >= 5) {
        const int j = 8 - layer;
        rl_patch_bwd_args pa = {};
        pa.B = B; pa.L = L; pa.C = C; pa.mode = 1;
        pa.g = g; pa.g2 = nullptr; pa.x = w.blk[i].y; pa.ln_w = P->ps[j][1]; pa.w = P->ps[j][0]; pa.u = w.ps_u[j];
        before_main();
        pa.dx = rot(); pa.gsum = nullptr;
        pa.d_w = G->ps[j][0]; pa.d_ln_w = G->ps[j][1]; pa.d_ln_b = G->ps[j][2];
        RlDet* d = det_on(w.det_patch, w.det_patch_n);
        if ((rc = rl_patch_bwd_main(&pa, st_main, d))) return rc;
        if ((rc = fork_grads(rl_patch_bwd_has_wgrad(&pa), d, [&](cudaStream_t q) { return rl_patch_bwd_wgrad(&pa, q, d); })))
          return rc;
        ++n;
        g = pa.dx;
      } else if (layer < 4) {
        g_extra_for_pm = w.gskip[layer + 1];       // skip consumer (ps / x_mid) gradient of pm_out[layer]
        rl_patch_bwd_args pa = {};
        pa.B = B; pa.L = L; pa.C = C; pa.mode = 0;
        pa.g = g; pa.g2 = g_extra_for_pm; pa.x = w.blk[i].y; pa.ln_w = P->pm[layer][1]; pa.w = P->pm[layer][0];
        pa.u = w.pm_u[layer];
        before_main();
        pa.dx = rot(); pa.gsum = w.gsum;
        pa.d_w = G->pm[layer][0]; pa.d_ln_w = G->pm[layer][1]; pa.d_ln_b = G->pm[layer][2];
        RlDet* d = det_on(w.det_patch, w.det_patch_n);
        if ((rc = rl_patch_bwd_main(&pa, st_main, d))) return rc;
        if ((rc = fork_grads(rl_patch_bwd_has_wgrad(&pa), d, [&](cudaStream_t q) { return rl_patch_bwd_wgrad(&pa, q, d); })))
          return rc;
        ++n;
        g = pa.dx;
      }
      // layer 4 ("transformer"): y9 = blk9(...) + x4; the x4 part is g itself, kept in gskip[4] below
    }
    const bool has_rw = rwi >= 0 && P->table[rwi] != nullptr;
    rl_ffn_bwd_args fa = {};
    fa.B = B; fa.L = L; fa.C = C; fa.le_mode = cfg->le_mode; fa.flags = RL_F_PRENORM | RL_F_RESIDUAL;
    fa.g = g; fa.x = w.blk[i].xa; fa.ln_w = bp[RL_BLK_LN2W]; fa.ln_b = bp[RL_BLK_LN2B];
    fa.w1 = bp[RL_BLK_W1]; fa.w2 = bp[RL_BLK_W2]; fa.lew = bp[RL_BLK_LEW]; fa.h = w.blk[i].h;
    before_main();
    fa.dx = rot(); fa.dh = w.dh[set]; fa.g2 = w.g2[set]; fa.u = w.uf[set];
    fa.d_ln_w = bg[RL_BLK_LN2W]; fa.d_ln_b = bg[RL_BLK_LN2B]; fa.d_w1 = bg[RL_BLK_W1]; fa.d_b1 = bg[RL_BLK_B1];
    fa.d_w2 = bg[RL_BLK_W2]; fa.d_b2 = bg[RL_BLK_B2]; fa.d_lew = bg[RL_BLK_LEW];
    RlDet* dfa = det_on(w.det_ffn[set], w.det_ffn_n);
    if ((rc = rl_ffn_bwd_main(&fa, st_main, dfa))) return rc;
    if ((rc = fork_grads(rl_ffn_bwd_has_wgrad(&fa), dfa, [&](cudaStream_t q) { return rl_ffn_bwd_wgrad(&fa, q, dfa); })))
      return rc;
    ++n;
    g = fa.dx;

    rl_attn_bwd_args aa = {};
    aa.B = B; aa.L = L; aa.C = C; aa.H = H;
    aa.W = has_rw ? kRwWindow[rwi] : 0;
    aa.c0 = has_rw ? (L - aa.W) / 2 : 0;
    aa.flags = RL_F_PRENORM | RL_F_RESIDUAL;
    aa.g = g; aa.x = block_input(i); aa.pe = cfg->pe[s];
    aa.ln_w = bp[RL_BLK_LN1W]; aa.ln_b = bp[RL_BLK_LN1B];
    aa.wq = bp[RL_BLK_WQ]; aa.wkv = bp[RL_BLK_WKV]; aa.wp = bp[RL_BLK_WP];
    aa.table = has_rw ? P->table[rwi] : nullptr;
    aa.q = w.blk[i].q; aa.k = w.blk[i].k; aa.v = w.blk[i].v; aa.o = w.blk[i].o; aa.lse = w.blk[i].lse;
    // where does dL/d(block input) go?  first block of an up layer (or of the mid layers) produces a
    // gradient that is also the U-skip gradient of a pm output, so it gets a dedicated buffer.
    before_main();
    float* dst;
    if (i % 2 == 0 && layer >= 5) dst = w.gskip[9 - layer];       // layer 5 -> gskip[4] (x_mid), 6 -> [3], 7 -> [2], 8 -> [1]
    else if (i == 0) dst = w.gfirst;                              // dL/d(stem output) through the blocks
    else dst = rot();
    aa.dx = dst; aa.dqkv = w.dqkv[set]; aa.u = w.ua[set];
    aa.d_ln_w = bg[RL_BLK_LN1W]; aa.d_ln_b = bg[RL_BLK_LN1B];
    aa.d_wq = bg[RL_BLK_WQ]; aa.d_bq = bg[RL_BLK_BQ]; aa.d_wkv = bg[RL_BLK_WKV]; aa.d_bkv = bg[RL_BLK_BKV];
    aa.d_wp = bg[RL_BLK_WP]; aa.d_bp = bg[RL_BLK_BP];
    aa.d_table = has_rw ? G->table[rwi] : nullptr;
    RlDet* daa = det_on(w.det_attn[set], w.det_attn_n);
    if ((rc = rl_attn_bwd_main(&aa, st_main, daa))) return rc;
    if ((rc = fork_grads(rl_attn_bwd_has_wgrad(&aa), daa, [&](cudaStream_t q) { return rl_attn_bwd_wgrad(&aa, q, daa); })))
      return rc;
    ++n;
    g = dst;
  }
  if (use_side && last_side >= 0) cudaStreamWaitEvent(st_main, sc->ev_side[last_side], 0);   // join
  // g = dL/d(x0) through the blocks; the final skip adds gx0 (transformer.py:665)
  rl_stem_bwd_args sb = {};
  sb.B = B; sb.L = L0; sb.training = cfg->training;
  sb.g = g; sb.g2 = w.gx0; sb.x = x; sb.conv_w = P->stem[0]; sb.conv_b = P->stem[1]; sb.bn_w = P->stem[2];
  sb.running_mean = cfg->running_mean; sb.running_var = cfg->running_var; sb.stats = cfg->bn_stats;
  sb.sums = cfg->bn_stats + 32; sb.partials = w.partials; sb.dx = nullptr;
  sb.d_conv_w = G->stem[0]; sb.d_conv_b = G->stem[1]; sb.d_bn_w = G->stem[2]; sb.d_bn_b = G->stem[3];
  sb.eps = 1e-5f;
  return ralenet_stem_bwd_stats(&sb, stream);
}

extern "C" int ralenet_net_bwd_stem(const rl_net_cfg* cfg, const rl_net_ptrs* P, const rl_net_ptrs* G, const float* x,
                                    float* dx, void* stream) {
  if (int rc = check_cfg(cfg, P)) return rc;
  RL_REQUIRE(G && x, RL_ERR_NULL, "net_bwd_stem: NULL argument");
  const int B = cfg->B, L0 = cfg->L0;
  const Ws w = carve((float*)cfg->ws, B, L0, 1, cfg->flags);
  const float* g = w.gfirst;
  rl_stem_bwd_args sb = {};
  sb.B = B; sb.L = L0; sb.training = cfg->training;
  sb.g = g; sb.g2 = w.gx0; sb.x = x; sb.conv_w = P->stem[0]; sb.conv_b = P->stem[1]; sb.bn_w = P->stem[2];
  sb.running_mean = cfg->running_mean; sb.running_var = cfg->running_var; sb.stats = cfg->bn_stats;
  sb.sums = cfg->bn_stats + 32; sb.partials = w.partials; sb.dx = dx;
  sb.d_conv_w = G->stem[0]; sb.d_conv_b = G->stem[1]; sb.d_bn_w = G->stem[2]; sb.d_bn_b = G->stem[3];
  sb.eps = 1e-5f;
  RlDet det = {w.det_ends, w.det_ends_n, 0, {}, 0};
  return rl_stem_bwd_apply(&sb, (cudaStream_t)stream, (cfg->flags & RL_NET_DETERMINISTIC) ? &det : nullptr);
}
