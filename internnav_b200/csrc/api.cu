// extern "C" surface of libn1b200.so (include/n1b200.h).  Exceptions stop here and become error codes.
#include <string.h>

#include <string>

#include "../../include/n1b200.h"
#include "n1_ops.h"
#include "resize.h"
#include "bwd_kernels.h"
#include "s1_model.h"
#include "s2_model.h"
#include "weights.h"

using namespace n1;

struct n1_ctx {
  int device = 0;
  S1Model s1;
  S2Model s2;
};
struct n1_vit_plan_s {
  VitPlan* p;
};
struct n1_llm_plan_s {
  LlmPlan* p;
};
struct n1_resize_plan_s {
  ResizePlan* p;
};

namespace {

thread_local std::string g_err;

template <typename F>
int guard(F&& f) {
  try {
    f();
    return N1_OK;
  } catch (const Error& e) {
    g_err = e.what();
    return e.code;
  } catch (const std::exception& e) {
    g_err = e.what();
    return N1_ERR_UNKNOWN;
  } catch (...) {
    g_err = "unknown error";
    return N1_ERR_UNKNOWN;
  }
}

void require_device(int device) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) throw Error(N1_ERR_NO_DEVICE, "no CUDA device visible; n1b200 has no CPU fallback");
  if (device < 0 || device >= n) throw Error(N1_ERR_NO_DEVICE, "device index out of range");
  cudaDeviceProp p;
  N1_CUDA(cudaGetDeviceProperties(&p, device));
  if (p.major != 10) throw Error(N1_ERR_NO_DEVICE, std::string("device is sm_") + std::to_string(p.major) + std::to_string(p.minor) + "; n1b200 kernels are sm_100a only");
}

void use(n1_handle h) {
  if (!h) throw Error(N1_ERR_ARG, "null handle");
  N1_CUDA(cudaSetDevice(h->device));
}

WeightSource to_source(const n1_tensor_desc* t, int n) {
  WeightSource ws;
  for (int i = 0; i < n; ++i) {
    if (!t[i].name || !t[i].data) throw Error(N1_ERR_WEIGHT, "tensor descriptor with null name/data");
    SrcTensor s;
    s.data = t[i].data;
    s.dtype = t[i].dtype;
    if (s.dtype != N1_F32 && s.dtype != N1_BF16) throw Error(N1_ERR_WEIGHT, std::string("unsupported dtype for ") + t[i].name);
    for (int d = 0; d < t[i].ndim && d < 4; ++d) s.shape.push_back(t[i].shape[d]);
    ws.add(t[i].name, s);
  }
  return ws;
}

inline cudaStream_t S(void* s) { return static_cast<cudaStream_t>(s); }
inline const bf16* B16(const void* p) { return static_cast<const bf16*>(p); }
inline bf16* B16(void* p) { return static_cast<bf16*>(p); }

}  // namespace

extern "C" {

const char* n1_version(void) { return "n1b200 0.1 (sm_100a)"; }

const char* n1_last_error(void) { return g_err.c_str(); }

int n1_device_ok(int device) {
  try {
    require_device(device);
    return 1;
  } catch (const std::exception& e) {
    g_err = e.what();
    return 0;
  }
}

int n1_create(n1_handle* out, int device) {
  return guard([&] {
    if (!out) throw Error(N1_ERR_ARG, "null out pointer");
    require_device(device);
    N1_CUDA(cudaSetDevice(device));
    n1_ctx* c = new n1_ctx();
    c->device = device;
    *out = c;
  });
}

void n1_destroy(n1_handle h) {
  if (!h) return;
  cudaSetDevice(h->device);
  delete h;
}

int n1_s1_load(n1_handle h, const n1_s1_dims* d, const n1_tensor_desc* tensors, int n, void* stream) {
  return guard([&] {
    use(h);
    if (!d || !tensors || n <= 0) throw Error(N1_ERR_ARG, "n1_s1_load: null dims/tensors");
    S1Dims dims;
    dims.D = d->token_dim, dims.heads = d->heads, dims.layers = d->layers, dims.T = d->predict_size;
    dims.frames = d->memory_size, dims.vlm_dim = d->vlm_token_dim, dims.n_query = d->n_query;
    h->s1.load(to_source(tensors, n), dims, S(stream));
  });
}

int n1_navdp_policy_load(n1_handle h, const n1_navdp_policy_dims* d, const n1_tensor_desc* tensors, int n, void* stream) {
  return guard([&] {
    use(h);
    if (!d || !tensors || n <= 0) throw Error(N1_ERR_ARG, "n1_navdp_policy_load: null dims/tensors");
    S1Dims dims;
    dims.D = d->token_dim, dims.heads = d->heads, dims.layers = d->layers, dims.T = d->predict_size;
    dims.frames = d->memory_size, dims.frames_depth = d->depth_frames, dims.goal_slots = d->goal_slots;
    dims.ddpm_steps = d->ddpm_steps, dims.standalone = 1, dims.vlm_dim = 0, dims.n_query = 0;
    h->s1.load(to_source(tensors, n), dims, S(stream));
  });
}

int n1_navdp_critic(n1_handle h, void* ws, size_t ws_bytes, const float* traj, const void* rgbd, float* critic, int B, int Ns,
                    int T, void* stream) {
  return guard([&] {
    use(h);
    h->s1.navdp_critic(ws, ws_bytes, traj, B16(rgbd), critic, B, Ns, T, S(stream));
  });
}

size_t n1_workspace_bytes(n1_handle h, int op, int B, int Ns, int T) {
  size_t r = 0;
  guard([&] {
    if (!h) throw Error(N1_ERR_ARG, "null handle");
    switch (op) {
      case N1_OP_RGBD: r = h->s1.ws_rgbd(B); break;
      case N1_OP_GOAL: r = h->s1.ws_goal(B); break;
      case N1_OP_DENOISE: r = h->s1.ws_denoise(B, Ns, T); break;
      default: throw Error(N1_ERR_ARG, "unknown op");
    }
  });
  return r;
}

int n1_rgbd_encode(n1_handle h, void* ws, size_t ws_bytes, const float* rgb, const float* depth, void* out, int B,
                   void* stream) {
  return guard([&] {
    use(h);
    h->s1.rgbd_encode(ws, ws_bytes, rgb, depth, B16(out), B, S(stream));
  });
}

int n1_goal_compress(n1_handle h, void* ws, size_t ws_bytes, const void* latents, void* goal, int B, void* stream) {
  return guard([&] {
    use(h);
    h->s1.goal_compress(ws, ws_bytes, B16(latents), B16(goal), B, S(stream));
  });
}

int n1_navdp_eps(n1_handle h, void* ws, size_t ws_bytes, const float* x_t, const int32_t* timesteps, int t_scalar,
                 const void* goal, const void* rgbd, float* eps, int B, int Ns, int T, void* stream) {
  return guard([&] {
    use(h);
    h->s1.navdp_eps(ws, ws_bytes, x_t, timesteps, t_scalar, B16(goal), B16(rgbd), eps, B, Ns, T, S(stream));
  });
}

int n1_navdp_sample(n1_handle h, void* ws, size_t ws_bytes, const void* goal, const void* rgbd, const float* x_init,
                    const float* step_noise, float* traj_out, int B, int Ns, int T, int K, void* stream) {
  return guard([&] {
    use(h);
    h->s1.navdp_sample(ws, ws_bytes, B16(goal), B16(rgbd), x_init, step_noise, traj_out, B, Ns, T, K, S(stream));
  });
}

int n1_ddpm_tables(int K, float* out_host) {
  return guard([&] {
    if (K <= 0 || !out_host) throw Error(N1_ERR_ARG, "n1_ddpm_tables: bad arguments");
    std::vector<DdpmCoef> c;
    S1Model::ddpm_tables(K, c);
    for (int i = 0; i < K; ++i) {
      out_host[i * 5 + 0] = c[i].sqrt_one_minus_acp, out_host[i * 5 + 1] = c[i].inv_sqrt_acp;
      out_host[i * 5 + 2] = c[i].c0, out_host[i * 5 + 3] = c[i].c1, out_host[i * 5 + 4] = c[i].sigma;
    }
  });
}

int n1_s2_load(n1_handle h, const n1_s2_dims* d, const n1_tensor_desc* tensors, int n, void* stream) {
  return guard([&] {
    use(h);
    if (!d || !tensors || n <= 0) throw Error(N1_ERR_ARG, "n1_s2_load: null dims/tensors");
    S2Dims x;
    x.v_depth = d->v_depth, x.v_hidden = d->v_hidden, x.v_heads = d->v_heads, x.v_inter = d->v_inter;
    x.v_patch = d->v_patch, x.v_tpatch = d->v_tpatch, x.v_merge = d->v_merge, x.v_window = d->v_window, x.v_out = d->v_out;
    x.n_fullatt = d->n_fullatt;
    if (x.n_fullatt < 0 || x.n_fullatt > 16) throw Error(N1_ERR_ARG, "n_fullatt out of range");
    for (int i = 0; i < 16; ++i) x.fullatt[i] = d->fullatt[i];
    x.layers = d->layers, x.hidden = d->hidden, x.heads = d->heads, x.kv_heads = d->kv_heads, x.head_dim = d->head_dim;
    x.inter = d->inter, x.vocab = d->vocab, x.rms_eps = d->rms_eps, x.rope_theta = d->rope_theta;
    for (int i = 0; i < 3; ++i) x.mrope[i] = d->mrope[i];
    x.n_query = d->n_query;
    h->s2.load(to_source(tensors, n), x, S(stream));
  });
}

int n1_vit_plan_create(n1_handle h, const int32_t* grid, int n_img, n1_vit_plan* out, void* stream) {
  return guard([&] {
    use(h);
    if (!grid || n_img <= 0 || !out) throw Error(N1_ERR_ARG, "n1_vit_plan_create: bad arguments");
    n1_vit_plan_s* w = new n1_vit_plan_s();
    try {
      w->p = h->s2.make_vit_plan(grid, n_img, S(stream));
    } catch (...) {
      delete w;
      throw;
    }
    *out = w;
  });
}
void n1_vit_plan_destroy(n1_vit_plan p) {
  if (!p) return;
  delete p->p;
  delete p;
}
int64_t n1_vit_plan_patches(n1_vit_plan p) { return p ? p->p->host.n_patches : 0; }

int n1_llm_plan_create(n1_handle h, const int32_t* ids, const int32_t* lens, int B, const int32_t* grid, int n_img,
                       n1_llm_plan* out, void* stream) {
  return guard([&] {
    use(h);
    if (!ids || !lens || B <= 0 || !out) throw Error(N1_ERR_ARG, "n1_llm_plan_create: bad arguments");
    n1_llm_plan_s* w = new n1_llm_plan_s();
    try {
      w->p = h->s2.make_llm_plan(ids, lens, B, grid, n_img, S(stream));
    } catch (...) {
      delete w;
      throw;
    }
    *out = w;
  });
}
void n1_llm_plan_destroy(n1_llm_plan p) {
  if (!p) return;
  delete p->p;
  delete p;
}
int64_t n1_llm_plan_tokens(n1_llm_plan p) { return p ? p->p->tokens : 0; }
int64_t n1_llm_plan_image_tokens(n1_llm_plan p) { return p ? p->p->n_image_tokens : 0; }
int n1_llm_plan_positions(n1_llm_plan p, int32_t* pos3, int32_t* delta) {
  return guard([&] {
    if (!p) throw Error(N1_ERR_ARG, "null plan");
    if (pos3) memcpy(pos3, p->p->h_pos3.data(), p->p->h_pos3.size() * sizeof(int32_t));
    if (delta) memcpy(delta, p->p->h_delta.data(), p->p->h_delta.size() * sizeof(int32_t));
  });
}

size_t n1_vit_workspace_bytes(n1_handle h, n1_vit_plan p) {
  size_t r = 0;
  guard([&] {
    if (!h || !p) throw Error(N1_ERR_ARG, "null handle/plan");
    r = h->s2.ws_vit(*p->p);
  });
  return r;
}
size_t n1_llm_workspace_bytes(n1_handle h, n1_llm_plan p) {
  size_t r = 0;
  guard([&] {
    if (!h || !p) throw Error(N1_ERR_ARG, "null handle/plan");
    r = h->s2.ws_llm(*p->p);
  });
  return r;
}

int n1_qwen_vit(n1_handle h, n1_vit_plan p, void* ws, size_t ws_bytes, const void* pixels, void* out, void* stream) {
  return guard([&] {
    use(h);
    if (!p) throw Error(N1_ERR_ARG, "null plan");
    h->s2.vit_forward(*p->p, ws, ws_bytes, B16(pixels), B16(out), S(stream));
  });
}
int n1_llm_prefill(n1_handle h, n1_llm_plan p, void* ws, size_t ws_bytes, const void* image_feats, void* latents,
                   void* stream) {
  return guard([&] {
    use(h);
    if (!p) throw Error(N1_ERR_ARG, "null plan");
    h->s2.llm_prefill(*p->p, ws, ws_bytes, B16(image_feats), B16(latents), S(stream));
  });
}

int n1_gen_plan_create(n1_handle h, const int32_t* ids, const int32_t* lens, int B, const int32_t* grid, int n_img,
                       int max_new_tokens, n1_llm_plan* out, void* stream) {
  return guard([&] {
    use(h);
    if (!ids || !lens || B <= 0 || !out || max_new_tokens < 1) throw Error(N1_ERR_ARG, "n1_gen_plan_create: bad arguments");
    n1_llm_plan_s* w = new n1_llm_plan_s();
    try {
      w->p = h->s2.make_llm_plan(ids, lens, B, grid, n_img, S(stream), max_new_tokens);
    } catch (...) {
      delete w;
      throw;
    }
    *out = w;
  });
}
size_t n1_generate_workspace_bytes(n1_handle h, n1_llm_plan p) {
  size_t r = 0;
  guard([&] {
    if (!h || !p) throw Error(N1_ERR_ARG, "null handle/plan");
    r = h->s2.ws_generate(*p->p);
  });
  return r;
}
int n1_s2_has_lm_head(n1_handle h) { return h && h->s2.has_lm_head() ? 1 : 0; }
int n1_llm_generate(n1_handle h, n1_llm_plan p, void* ws, size_t ws_bytes, const void* image_feats,
                    const int32_t* eos, int n_eos, int32_t pad_id, int32_t* tokens, int32_t* lens, void* latents,
                    int32_t* passes, void* stream) {
  return guard([&] {
    use(h);
    if (!p) throw Error(N1_ERR_ARG, "null plan");
    if (n_eos < 0 || n_eos > 4 || (n_eos > 0 && !eos)) throw Error(N1_ERR_ARG, "n1_llm_generate: 0..4 eos ids");
    GenResult r;
    r.tokens = tokens, r.lens = lens;
    h->s2.llm_generate(*p->p, ws, ws_bytes, B16(image_feats), eos, n_eos, pad_id, r, B16(latents), S(stream));
    if (passes) *passes = r.steps;
  });
}

int n1_resize_plan_create(int in_h, int in_w, int out_h, int out_w, n1_resize_plan* out, void* stream) {
  return guard([&] {
    if (!out || in_h <= 0 || in_w <= 0 || out_h <= 0 || out_w <= 0) throw Error(N1_ERR_ARG, "n1_resize_plan_create: bad sizes");
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) throw Error(N1_ERR_NO_DEVICE, "no CUDA device visible; n1b200 has no CPU fallback");
    require_device(dev);
    n1_resize_plan_s* w = new n1_resize_plan_s();
    try {
      w->p = new ResizePlan(in_h, in_w, out_h, out_w, S(stream));
    } catch (...) {
      delete w;
      throw;
    }
    *out = w;
  });
}
void n1_resize_plan_destroy(n1_resize_plan p) {
  if (!p) return;
  delete p->p;
  delete p;
}
size_t n1_resize_workspace_bytes(n1_resize_plan p, int n, int is_float) {
  return p && n > 0 ? p->p->workspace_bytes(n, is_float ? 1 : 3, is_float != 0) : 0;
}
int n1_resize_rgb_u8(n1_resize_plan p, const void* src, int n, void* dst_f32, void* dst_u8, void* ws, size_t ws_bytes,
                     void* stream) {
  return guard([&] {
    if (!p) throw Error(N1_ERR_ARG, "null plan");
    if (ws_bytes < p->p->workspace_bytes(n, 3, false)) throw Error(N1_ERR_WORKSPACE, "n1_resize_rgb_u8: workspace too small");
    resize_rgb_u8(*p->p, static_cast<const uint8_t*>(src), n, static_cast<float*>(dst_f32), static_cast<uint8_t*>(dst_u8),
                  ws, S(stream));
  });
}
int n1_resize_f32(n1_resize_plan p, const void* src, int n, float mul, float clip_max, void* dst, void* ws,
                  size_t ws_bytes, void* stream) {
  return guard([&] {
    if (!p) throw Error(N1_ERR_ARG, "null plan");
    if (ws_bytes < p->p->workspace_bytes(n, 1, true)) throw Error(N1_ERR_WORKSPACE, "n1_resize_f32: workspace too small");
    resize_f32(*p->p, static_cast<const float*>(src), n, mul, clip_max, static_cast<float*>(dst), ws, S(stream));
  });
}
int n1_resize_coeffs(int in_size, int out_size, int capacity_k, int32_t* bounds, double* weights, int32_t* fixed,
                     int32_t* ksize) {
  return guard([&] {
    if (!bounds || !weights || !fixed || !ksize) throw Error(N1_ERR_ARG, "n1_resize_coeffs: null outputs");
    ResizeCoeffs c;
    resize_coeffs(in_size, out_size, c);
    if (c.ksize > capacity_k) throw Error(N1_ERR_ARG, "n1_resize_coeffs: capacity_k < " + std::to_string(c.ksize));
    *ksize = c.ksize;
    memcpy(bounds, c.bounds.data(), c.bounds.size() * sizeof(int32_t));
    memcpy(weights, c.weights.data(), c.weights.size() * sizeof(double));
    memcpy(fixed, c.fixed.data(), c.fixed.size() * sizeof(int32_t));
  });
}

size_t n1_rgb_tokens_workspace_bytes(n1_handle h, int B) {
  size_t r = 0;
  guard([&] {
    if (!h || B <= 0) throw Error(N1_ERR_ARG, "null handle / B <= 0");
    r = h->s1.ws_rgb_tokens(B);
  });
  return r;
}
int n1_rgb_tokens(n1_handle h, void* ws, size_t ws_bytes, const float* rgb, void* mem, int B, void* stream) {
  return guard([&] {
    use(h);
    h->s1.rgb_tokens(ws, ws_bytes, rgb, B16(mem), B, S(stream));
  });
}
int n1_s2_set_latent_queries(n1_handle h, const void* src, void* stream) {
  return guard([&] {
    use(h);
    h->s2.set_latent_queries(B16(src), S(stream));
  });
}
size_t n1_s2_train_workspace_bytes(n1_handle h, n1_llm_plan p) {
  size_t r = 0;
  guard([&] {
    if (!h || !p) throw Error(N1_ERR_ARG, "null handle/plan");
    r = h->s2.ws_train(*p->p);
  });
  return r;
}
int n1_s2_train_forward(n1_handle h, n1_llm_plan p, void* ws, size_t ws_bytes, const void* image_feats, void* states,
                        void* stream) {
  return guard([&] {
    use(h);
    if (!p) throw Error(N1_ERR_ARG, "null plan");
    h->s2.train_forward(*p->p, ws, ws_bytes, B16(image_feats), B16(states), S(stream));
  });
}
int n1_s2_train_backward(n1_handle h, n1_llm_plan p, void* ws, size_t ws_bytes, const void* grad_states, void* grad_latent,
                         void* stream) {
  return guard([&] {
    use(h);
    if (!p) throw Error(N1_ERR_ARG, "null plan");
    h->s2.train_backward(*p->p, ws, ws_bytes, B16(grad_states), static_cast<float*>(grad_latent), S(stream));
  });
}
int n1_op_transpose(const void* in, int rows, int cols, int ld_in, void* out, int ld_out, int rows_pad, void* stream) {
  return guard([&] { transpose_bf16(B16(in), rows, cols, ld_in, B16(out), ld_out, rows_pad, S(stream)); });
}
int n1_op_colsum(const void* a, const void* b, int rows, int cols, int ld_a, int ld_b, void* out, int accumulate, void* stream) {
  return guard([&] { colsum_bf16(B16(a), B16(b), rows, cols, ld_a, ld_b, static_cast<float*>(out), accumulate, S(stream)); });
}
int n1_op_norm_bwd(const void* dy, int ld_dy, const void* x, int ld_x, const void* w, const void* rg, int ld_rg, void* dx,
                   int ld_dx, void* dw, void* db, int rows, int D, float eps, int rms, int accumulate, void* stream) {
  return guard([&] {
    norm_bwd(B16(dy), ld_dy, B16(x), ld_x, static_cast<const float*>(w), B16(rg), ld_rg, B16(dx), ld_dx,
             static_cast<float*>(dw), static_cast<float*>(db), rows, D, eps, rms, accumulate, S(stream));
  });
}
int n1_op_act_fwd(const void* pre, void* out, int64_t n, int act, void* stream) {
  return guard([&] { act_fwd(B16(pre), B16(out), n, act, S(stream)); });
}
int n1_op_act_bwd(const void* pre, const void* dy, void* out, int64_t n, int act, void* stream) {
  return guard([&] { act_bwd(B16(pre), B16(dy), B16(out), n, act, S(stream)); });
}
int n1_op_swiglu_bwd(const void* pre, const void* dact, void* dpre, int64_t rows, int inter, void* stream) {
  return guard([&] { swiglu_bwd(B16(pre), B16(dact), B16(dpre), rows, inter, S(stream)); });
}
int n1_op_rope_transposed(void* x, int ld, const void* cs, int64_t rows, int heads, int head_dim, void* stream) {
  return guard([&] { rope_transposed(B16(x), ld, static_cast<const float2*>(cs), rows, heads, head_dim, S(stream)); });
}
int n1_op_attention_bwd(const void* q, const void* k, const void* v, const void* o, const void* dout, void* dq, void* dk,
                        void* dv, int ldq, int ldk, int ldv, int ldo, int lddo, int lddq, int heads_q, int heads_kv, int hd,
                        int batch, int seq_q, int seq_k, const void* cu_q, const void* cu_k, int max_seq_q, int kv_div,
                        int causal, float scale, const void* k_len, int k_slot, void* stream) {
  return guard([&] {
    AttnBwdParams p = {};
    p.f.q = B16(q), p.f.k = B16(k), p.f.v = B16(v), p.f.o = const_cast<bf16*>(B16(o));
    p.f.ldq = ldq, p.f.ldk = ldk, p.f.ldv = ldv, p.f.ldo = ldo;
    p.f.heads_q = heads_q, p.f.heads_kv = heads_kv, p.f.hd = hd, p.f.batch = batch, p.f.seq_q = seq_q, p.f.seq_k = seq_k;
    p.f.cu_q = static_cast<const int*>(cu_q), p.f.cu_k = static_cast<const int*>(cu_k), p.f.max_seq_q = max_seq_q;
    p.f.kv_div = kv_div, p.f.causal = causal, p.f.scale = scale;
    p.f.k_len = static_cast<const int*>(k_len), p.f.k_slot = k_slot;
    p.dout = B16(dout), p.lddo = lddo, p.dq = B16(dq), p.lddq = lddq;
    p.dk = static_cast<float*>(dk), p.dv = static_cast<float*>(dv);
    attention_bwd(p, S(stream));
  });
}
int n1_op_dropout_add(const void* residual, const void* y, void* out, int64_t n, const void* rng, int site, double p,
                      void* stream) {
  return guard([&] {
    if (!residual || p <= 0.0) throw Error(N1_ERR_ARG, "n1_op_dropout_add: needs a residual and p > 0");
    dropout_apply(B16(y), B16(residual), B16(out), n, make_dropout(rng, site, p), S(stream));
  });
}
int n1_op_dropout_bwd(const void* dy, void* out, int64_t n, const void* rng, int site, double p, void* stream) {
  return guard([&] {
    if (p <= 0.0) throw Error(N1_ERR_ARG, "n1_op_dropout_bwd: p > 0");
    dropout_apply(B16(dy), nullptr, B16(out), n, make_dropout(rng, site, p), S(stream));
  });
}
int n1_op_dropout_mask(void* out_u8, int64_t n, const void* rng, int site, double p, void* stream) {
  return guard([&] {
    if (p <= 0.0) throw Error(N1_ERR_ARG, "n1_op_dropout_mask: p > 0");
    dropout_mask(static_cast<uint8_t*>(out_u8), n, make_dropout(rng, site, p), S(stream));
  });
}
int n1_op_act_fwd_dropout(const void* pre, void* out, int64_t n, int act, const void* rng, int site, double p, void* stream) {
  return guard([&] {
    if (p <= 0.0) throw Error(N1_ERR_ARG, "n1_op_act_fwd_dropout: p > 0");
    act_fwd_dropout(B16(pre), B16(out), n, act, make_dropout(rng, site, p), S(stream));
  });
}
int n1_op_act_bwd_dropout(const void* pre, const void* dy, void* out, int64_t n, int act, const void* rng, int site, double p,
                          void* stream) {
  return guard([&] {
    if (p <= 0.0) throw Error(N1_ERR_ARG, "n1_op_act_bwd_dropout: p > 0");
    act_bwd_dropout(B16(pre), B16(dy), B16(out), n, act, make_dropout(rng, site, p), S(stream));
  });
}
int n1_op_attention_dropout(const void* q, const void* k, const void* v, void* o, int ldq, int ldk, int ldv, int ldo, int heads,
                            int head_dim, int batch, int seq_q, int seq_k, int causal, float scale, const void* rng, int site,
                            double p, void* stream) {
  return guard([&] {
    AttnParams a = {};
    a.q = B16(q), a.k = B16(k), a.v = B16(v), a.o = B16(o);
    a.ldq = ldq, a.ldk = ldk, a.ldv = ldv, a.ldo = ldo;
    a.heads_q = a.heads_kv = heads, a.hd = head_dim, a.batch = batch, a.seq_q = seq_q, a.seq_k = seq_k;
    a.kv_div = 1, a.causal = causal, a.scale = scale;
    a.drop = make_dropout(rng, site, p);
    attention(a, S(stream));
  });
}
int n1_op_attention_bwd_dropout(const void* q, const void* k, const void* v, const void* o, const void* dout, void* dq,
                                void* dk, void* dv, int ldq, int ldk, int ldv, int ldo, int lddo, int lddq, int heads,
                                int head_dim, int batch, int seq_q, int seq_k, int causal, float scale, const void* rng,
                                int site, double p, void* stream) {
  return guard([&] {
    AttnBwdParams a = {};
    a.f.q = B16(q), a.f.k = B16(k), a.f.v = B16(v), a.f.o = const_cast<bf16*>(B16(o));
    a.f.ldq = ldq, a.f.ldk = ldk, a.f.ldv = ldv, a.f.ldo = ldo;
    a.f.heads_q = a.f.heads_kv = heads, a.f.hd = head_dim, a.f.batch = batch, a.f.seq_q = seq_q, a.f.seq_k = seq_k;
    a.f.kv_div = 1, a.f.causal = causal, a.f.scale = scale;
    a.f.drop = make_dropout(rng, site, p);
    a.dout = B16(dout), a.lddo = lddo, a.dq = B16(dq), a.lddq = lddq;
    a.dk = static_cast<float*>(dk), a.dv = static_cast<float*>(dv);
    attention_bwd(a, S(stream));
  });
}
int n1_traj_to_actions(const void* traj, int B, int Ns, int T, double turn_angle_rad, double step_size, int lookahead,
                       int max_actions, int cap, int32_t* ids, int32_t* count, double* mean_path, void* stream) {
  return guard([&] {
    traj_to_actions(static_cast<const float*>(traj), B, Ns, T, turn_angle_rad, step_size, lookahead, max_actions, cap, ids,
                    count, mean_path, S(stream));
  });
}
int n1_op_sgemm(const void* A, int lda, int trans_a, const void* B, int ldb, int trans_b, void* C, int ldc, int M, int N, int K,
                int accumulate, void* stream) {
  return guard([&] {
    sgemm_small(static_cast<const float*>(A), lda, trans_a, static_cast<const float*>(B), ldb, trans_b, static_cast<float*>(C),
                ldc, M, N, K, accumulate, S(stream));
  });
}
size_t n1_op_wgrad_workspace_bytes(int M, int No, int Ko) { return wgrad_tn_workspace_bytes(M, No, Ko); }
int n1_op_wgrad(const void* dy, int ld_dy, const void* x, int ld_x, int M, int No, int Ko, void* out, int accumulate, void* ws,
                size_t ws_bytes, void* stream) {
  return guard([&] {
    wgrad_tn(B16(dy), ld_dy, B16(x), ld_x, M, No, Ko, static_cast<float*>(out), accumulate, ws, ws_bytes, S(stream));
  });
}
int n1_op_scale_cols(const void* x, int ld_x, const void* gamma, const void* add, int ld_add, void* out, int ld_out,
                     int64_t rows, int cols, void* stream) {
  return guard([&] {
    scale_cols(B16(x), ld_x, static_cast<const float*>(gamma), B16(add), ld_add, B16(out), ld_out, rows, cols, S(stream));
  });
}
int n1_op_patchify_depth(const void* img, void* out, int n_img, int ldk, void* stream) {
  return guard([&] {
    if (!img || !out || n_img <= 0 || ldk < 196 || ldk % 8) throw Error(N1_ERR_ARG, "n1_op_patchify_depth: bad arguments");
    patchify_depth(static_cast<const float*>(img), B16(out), n_img, ldk, S(stream));
  });
}
int n1_op_adamw(void* master, void* working, const void* grad, void* m, void* v, int64_t n, float lr, float beta1,
                float beta2, float eps, float weight_decay, int step, void* stream) {
  return guard([&] {
    adamw_step(static_cast<float*>(master), B16(working), static_cast<const float*>(grad), static_cast<float*>(m),
               static_cast<float*>(v), n, lr, beta1, beta2, eps, weight_decay, step, S(stream));
  });
}

int n1_rope_index(const int32_t* ids, int len, const int32_t* grid, int n_img, int merge, int32_t* pos3,
                  int32_t* delta) {
  return guard([&] {
    if (!ids || len <= 0 || !pos3) throw Error(N1_ERR_ARG, "n1_rope_index: bad arguments");
    std::vector<int> p;
    int cursor = 0, d = 0;
    rope_index_one(ids, len, grid, n_img, merge, cursor, p, d);
    memcpy(pos3, p.data(), p.size() * sizeof(int32_t));
    if (delta) *delta = d;
  });
}
int n1_vit_window_index(const int32_t* grid, int n_img, int merge, int window, int32_t* widx, int32_t* cu, int32_t* n_cu,
                        int32_t* pos_hw) {
  return guard([&] {
    if (!grid || n_img <= 0) throw Error(N1_ERR_ARG, "n1_vit_window_index: bad arguments");
    VitIndex v;
    vit_index(grid, n_img, merge, window, v);
    if (widx) memcpy(widx, v.window_index.data(), v.window_index.size() * sizeof(int32_t));
    if (cu) memcpy(cu, v.cu_window.data(), v.cu_window.size() * sizeof(int32_t));
    if (n_cu) *n_cu = (int32_t)v.cu_window.size();
    if (pos_hw) memcpy(pos_hw, v.pos_hw.data(), v.pos_hw.size() * sizeof(int32_t));
  });
}

void n1_prof_enable(int on) { prof_enable(on != 0); }

void n1_prof_add(int64_t gemm_launches, int64_t total_launches) {
  // a replayed CUDA graph launches the kernels captured in it without passing through the launchers: account for them
  prof_count_launch((int)(total_launches - gemm_launches));
  for (int64_t i = 0; i < gemm_launches; ++i) prof_count_gemm(0.0);
}

int n1_prof_read_shapes(int32_t* mnk, int64_t* count, double* ms, int cap) {
  int n = -1;
  guard([&] {
    if (!mnk || !count || !ms || cap <= 0) throw Error(N1_ERR_ARG, "n1_prof_read_shapes: bad arguments");
    n = prof_read_shapes(mnk, reinterpret_cast<long*>(count), ms, cap);
  });
  return n;
}

int n1_prof_read(double* gemm_ms, double* gemm_flops, int64_t* gemm_launches, int64_t* total_launches) {
  return guard([&] {
    ProfStats st = prof_read_and_reset();
    if (gemm_ms) *gemm_ms = st.gemm_ms;
    if (gemm_flops) *gemm_flops = st.gemm_flops;
    if (gemm_launches) *gemm_launches = st.gemm_launches;
    if (total_launches) *total_launches = st.total_launches;
  });
}

int n1_op_gemm(const void* A, int lda, const void* W, int ldw, void* out, int ldo, int M, int N, int K,
               const float* bias, const float* gamma, const void* residual, int ldr, int act, int out_fp32,
               void* stream) {
  return guard([&] {
    GemmEpilogue e;
    e.bias = bias, e.gamma = gamma, e.residual = B16(residual), e.ldr = ldr, e.act = act, e.out_fp32 = out_fp32;
    gemm_bf16(B16(A), lda, B16(W), ldw, out, ldo, M, N, K, e, S(stream));
  });
}

int n1_op_ff_block(const void* x, int ldx, const float* ln_w, const float* ln_b, float eps, const void* w1, const float* b1,
                   const void* w2, const float* b2, void* out, int ldo, int M, int cluster, void* stream) {
  return guard([&] {
    ff_block_384(B16(x), ldx, ln_w, ln_b, eps, B16(w1), b1, B16(w2), b2, B16(out), ldo, M, cluster, S(stream));
  });
}

int n1_op_mod_norm(const void* x, int ldx, const float* w, const void* mod, int ld_mod, int rows_per_group, const void* res,
                   int ldr, void* out, int ldo, int64_t rows, int D, float eps, int mode, void* stream) {
  return guard([&] {
    mod_norm(B16(x), ldx, w, B16(mod), ld_mod, rows_per_group, B16(res), ldr, B16(out), ldo, rows, D, eps, mode, S(stream));
  });
}
int n1_op_add(const void* a, const void* b, void* out, int64_t n, void* stream) {
  return guard([&] { add_bf16(B16(a), B16(b), B16(out), n, S(stream)); });
}
int n1_op_action_embed(const float* lat, const float* w, const float* b, const float* pos, void* out, int64_t rows, int T, int D,
                       void* stream) {
  return guard([&] { action_embed(lat, w, b, pos, B16(out), rows, T, D, S(stream)); });
}
int n1_op_cfg_euler(const void* pred, int ld, int64_t n, int cfg, float scale, float dt, float* lat, void* stream) {
  return guard([&] { cfg_euler(B16(pred), ld, n, cfg, scale, dt, lat, S(stream)); });
}
int n1_op_layernorm(const void* x, int ldx, void* y, int ldy, const float* w, const float* b, int rows, int D, float eps,
                    int rms, void* stream) {
  return guard([&] { layernorm(B16(x), ldx, B16(y), ldy, w, b, rows, D, eps, rms, S(stream)); });
}

int n1_op_attention(const void* q, const void* k, const void* v, void* o, int ldq, int ldk, int ldv, int ldo, int heads_q,
                    int heads_kv, int head_dim, int batch, int seq_q, int seq_k, const int32_t* cu_q,
                    const int32_t* cu_k, int max_seq_q, int kv_div, int causal, float scale, void* stream) {
  return guard([&] {
    AttnParams p = {};
    p.q = B16(q), p.k = B16(k), p.v = B16(v), p.o = B16(o);
    p.ldq = ldq, p.ldk = ldk, p.ldv = ldv, p.ldo = ldo;
    p.heads_q = heads_q, p.heads_kv = heads_kv, p.hd = head_dim, p.batch = batch;
    p.seq_q = seq_q, p.seq_k = seq_k, p.cu_q = cu_q, p.cu_k = cu_k, p.max_seq_q = max_seq_q;
    p.kv_div = kv_div < 1 ? 1 : kv_div, p.causal = causal, p.scale = scale;
    attention(p, S(stream));
  });
}

/* n1_op_attention with the row count of the packed buffers: lets var-len self-attention with head_dim 128 and <= 320
 * tokens per sequence take the tcgen05 kernel (attention_tc.cu), which addresses q / k / v through TMA tensor maps */
int n1_op_attention_ex(const void* q, const void* k, const void* v, void* o, int ldq, int ldk, int ldv, int ldo, int heads_q,
                       int heads_kv, int head_dim, int batch, const int32_t* cu_seqlens, int max_seq, int64_t total_rows,
                       int causal, float scale, int* used_tcgen05, void* stream) {
  return guard([&] {
    AttnParams p = {};
    p.q = B16(q), p.k = B16(k), p.v = B16(v), p.o = B16(o);
    p.ldq = ldq, p.ldk = ldk, p.ldv = ldv, p.ldo = ldo;
    p.heads_q = heads_q, p.heads_kv = heads_kv, p.hd = head_dim, p.batch = batch;
    p.cu_q = p.cu_k = cu_seqlens, p.max_seq_q = max_seq, p.total_rows = total_rows;
    p.kv_div = 1, p.causal = causal, p.scale = scale;
    if (used_tcgen05) *used_tcgen05 = (head_dim == 128 && attention_tc_supported(p)) ? 1 : 0;
    attention(p, S(stream));
  });
}

}  // extern "C"
