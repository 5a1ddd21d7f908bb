// Context management, GEMM dispatch and the three model pipelines of the hot path:
//   cir_vit_forward        VisionTransformer.forward                 src/vit.py:180-194
//   cir_stage1_encode      BLIP_Retrieval.img_txt_fusion(train=False) src/blip_stage1.py:67-88 -> src/med.py:685-821
//   cir_stage2_score       BLIP_NLVR.img_txt_fusion_val              src/blip_stage2.py:101-136 -> src/nlvr_encoder.py:777-909
// Each pipeline is a fixed sequence of kernel launches on the context's stream over a
// caller-provided workspace; nothing allocates or synchronises.
#include "common.cuh"

// rowops.cu internals
int cir_im2col16(cir_ctx* ctx, const float* img, void* out, int64_t B, int S);
int cir_vit_assemble(cir_ctx* ctx, const float* patch, const float* cls, const float* pos, float* x, int64_t B, int64_t N);
int cir_gather_cls(cir_ctx* ctx, const void* h, int64_t T, int64_t L, void* feats, float* feats_f32);
int cir_head_dot(cir_ctx* ctx, const float* hidden, const float* w, const float* b, float* scores, int64_t rows);

#include <algorithm>
#include <vector>
struct ProfState {
  std::vector<cudaEvent_t> ev;      // pairs: [2i] start, [2i+1] end
  std::vector<double> work;         // algorithmic FLOPs (GEMM, attention) or bytes (LayerNorm) of launch i
  std::vector<int> kind;            // CIR_PROF_*
  size_t used = 0;                  // pairs in use
};
void cir_prof_begin(cir_ctx* ctx, int kind, double work) {
  if (!ctx->profiling) return;
  ProfState* ps = (ProfState*)ctx->prof;
  if (ps->used * 2 + 2 > ps->ev.size()) {
    cudaEvent_t a, b;
    cudaEventCreate(&a); cudaEventCreate(&b);
    ps->ev.push_back(a); ps->ev.push_back(b);
    ps->work.push_back(0.0);
    ps->kind.push_back(0);
  }
  ps->work[ps->used] = work;
  ps->kind[ps->used] = kind;
  cudaEventRecord(ps->ev[ps->used * 2], ctx->stream);
}
void cir_prof_end(cir_ctx* ctx) {
  if (!ctx->profiling) return;
  ProfState* ps = (ProfState*)ctx->prof;
  cudaEventRecord(ps->ev[ps->used * 2 + 1], ctx->stream);
  ps->used++;
}
void cir_prof_gemm_begin(cir_ctx* ctx, double flops) { cir_prof_begin(ctx, CIR_PROF_GEMM, flops); }
void cir_prof_gemm_end(cir_ctx* ctx) { cir_prof_end(ctx); }

static thread_local char g_err[1024] = "";
void cir_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

extern "C" const char* cir_last_error(void) { return g_err; }
extern "C" int cir_version(void) { return 100; }

extern "C" int cir_create(cir_ctx** out, int device, int dtype) {
  CIR_CHECK_ARG(out != nullptr, "cir_create: out is NULL");
  CIR_CHECK_ARG(dtype == CIR_DTYPE_F32 || dtype == CIR_DTYPE_BF16, "cir_create: bad dtype %d", dtype);
  int ndev = 0;
  CIR_CUDA(cudaGetDeviceCount(&ndev));
  CIR_CHECK_ARG(device >= 0 && device < ndev, "cir_create: device %d out of range (have %d)", device, ndev);
  cudaDeviceProp prop;
  CIR_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    cir_set_error("cir_create: device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor);
    return CIR_EUNSUPPORTED;
  }
  CirDeviceGuard guard(device);      // initialise the device's primary context without changing the caller's current device
  CIR_CUDA(cudaFree(0));
  cir_ctx* c = new cir_ctx();
  c->device = device;
  c->dtype = dtype;
  c->gemm_impl = CIR_GEMM_AUTO;
  c->attn_impl = 0;
  c->gemm_pair = 1;
  c->gemm_force_pair = 0;
  c->prune_last = 1;
  c->dedup_first = 1;
  c->fuse_qkv = 1;
  c->stage1_tc = 1;
  c->gemm_tma_store = 1;
  c->func_attr_mask = 0;
  c->stream = 0;
  c->num_sms = prop.multiProcessorCount;
  c->launches = 0;
  c->encode_tiled = nullptr;
  c->profiling = 0;
  c->prof = new ProfState();
  *out = c;
  return CIR_OK;
}
extern "C" int cir_destroy(cir_ctx* ctx) {
  if (!ctx) return CIR_OK;
  ProfState* ps = (ProfState*)ctx->prof;
  for (cudaEvent_t e : ps->ev) cudaEventDestroy(e);
  delete ps;
  delete ctx;
  return CIR_OK;
}
extern "C" int cir_profile_gemm(cir_ctx* ctx, int enable) {
  ProfState* ps = (ProfState*)ctx->prof;
  ctx->profiling = enable ? 1 : 0;
  if (enable) ps->used = 0;
  return CIR_OK;
}
extern "C" int cir_profile_read(cir_ctx* ctx, int kind, double* total_ms, double* total_work, int64_t* launches) {
  CIR_ENTER(ctx);
  CIR_CHECK_ARG(kind >= 0 && kind < CIR_PROF_KINDS && total_ms && total_work && launches, "profile_read: bad argument");
  ProfState* ps = (ProfState*)ctx->prof;
  double ms = 0.0, wk = 0.0;
  int64_t n = 0;
  for (size_t i = 0; i < ps->used; i++) {
    if (ps->kind[i] != kind) continue;
    float t = 0.f;
    CIR_CUDA(cudaEventSynchronize(ps->ev[2 * i + 1]));
    CIR_CUDA(cudaEventElapsedTime(&t, ps->ev[2 * i], ps->ev[2 * i + 1]));
    ms += t; wk += ps->work[i]; n++;
  }
  *total_ms = ms; *total_work = wk; *launches = n;
  return CIR_OK;
}
extern "C" int cir_profile_gemm_read(cir_ctx* ctx, double* total_ms, double* total_flops, int64_t* launches) {
  return cir_profile_read(ctx, CIR_PROF_GEMM, total_ms, total_flops, launches);
}
extern "C" int cir_set_stream(cir_ctx* ctx, void* s) { ctx->stream = (cudaStream_t)s; return CIR_OK; }
extern "C" int cir_set_gemm_impl(cir_ctx* ctx, int impl) {
  CIR_CHECK_ARG(impl >= CIR_GEMM_AUTO && impl <= CIR_GEMM_TCGEN05_1CTA, "bad gemm impl %d", impl);
  CIR_CHECK_ARG(!(impl >= CIR_GEMM_TCGEN05 && ctx->dtype != CIR_DTYPE_BF16), "tcgen05 GEMM needs a bf16 context");
  ctx->gemm_pair = impl == CIR_GEMM_TCGEN05_1CTA ? 0 : 1;
  ctx->gemm_impl = impl == CIR_GEMM_TCGEN05_1CTA ? CIR_GEMM_TCGEN05 : impl;
  return CIR_OK;
}
extern "C" int cir_set_attention_impl(cir_ctx* ctx, int impl) {
  CIR_CHECK_ARG(impl >= 0 && impl <= 2, "bad attention impl %d", impl);
  ctx->attn_impl = impl;
  return CIR_OK;
}
extern "C" int cir_set_prune_last_layer(cir_ctx* ctx, int enable) { ctx->prune_last = enable ? 1 : 0; return CIR_OK; }
extern "C" int cir_set_dedup_first_layer(cir_ctx* ctx, int enable) { ctx->dedup_first = enable ? 1 : 0; return CIR_OK; }
extern "C" int cir_set_fuse_qkv_attention(cir_ctx* ctx, int enable) { ctx->fuse_qkv = enable ? 1 : 0; return CIR_OK; }
extern "C" int cir_set_stage1_tensor_cores(cir_ctx* ctx, int enable) { ctx->stage1_tc = enable ? 1 : 0; return CIR_OK; }
extern "C" int cir_set_gemm_tma_store(cir_ctx* ctx, int enable) { ctx->gemm_tma_store = enable ? 1 : 0; return CIR_OK; }
extern "C" int cir_get_dtype(const cir_ctx* ctx) { return ctx->dtype; }
extern "C" int64_t cir_launch_count(cir_ctx* ctx, int reset) {
  int64_t n = ctx->launches;
  if (reset) ctx->launches = 0;
  return n;
}

extern "C" int cir_gemm(cir_ctx* ctx, const cir_gemm_args* a) {
  CIR_ENTER(ctx);
  CIR_CHECK_ARG(a && a->A && a->W && a->C, "gemm: null operand");
  CIR_CHECK_ARG(a->M >= 0 && a->N >= 0 && a->K > 0 && a->batch >= 0, "gemm: bad shape M=%lld N=%lld K=%lld", (long long)a->M, (long long)a->N, (long long)a->K);
  const bool tc = ctx->dtype == CIR_DTYPE_BF16 && ctx->gemm_impl != CIR_GEMM_SIMT;
  return tc ? cir_gemm_tcgen05(ctx, a) : cir_gemm_simt(ctx, a);
}

// ------------------------------------------------------------------------------------------
namespace {

struct Bump {
  char* base; size_t off, cap; bool ok;
  Bump(void* p, size_t n) : base((char*)p), off(0), cap(n), ok(true) {}
  void* take(size_t bytes) {
    off = align_up(off, 256);
    void* r = base ? base + off : nullptr;
    off += bytes;
    if (base && off > cap) ok = false;
    return r;
  }
};

// thin wrapper: C[batch][M,N] = act(A W^T + bias) (+res)
int gemm(cir_ctx* ctx, const void* A, int64_t lda, int64_t a_bs, const void* W, int64_t ldw, int64_t w_bs, const float* bias,
         int64_t bias_bs, void* C, int64_t ldc, int64_t c_bs, int c_f32, const void* res, int64_t ldres, int64_t res_bs, int res_f32,
         int64_t M, int64_t N, int64_t K, int batch, int act) {
  cir_gemm_args g{};
  g.A = A; g.W = W; g.C = C; g.bias = bias; g.residual = res;
  g.M = M; g.N = N; g.K = K; g.lda = lda; g.ldw = ldw; g.ldc = ldc; g.ldres = ldres;
  g.a_bstride = a_bs; g.w_bstride = w_bs; g.c_bstride = c_bs; g.bias_bstride = bias_bs; g.res_bstride = res_bs;
  g.batch = batch; g.act = act; g.c_f32 = c_f32; g.res_f32 = res_f32;
  return cir_gemm(ctx, &g);
}

inline char* at(void* p, int64_t elems, size_t esz) { return (char*)p + elems * (int64_t)esz; }

// y = LayerNorm(A W^T + bias + res) with per-batch gamma/beta [batch][N=768], rows contiguous (ld = 768): GEMM into `pre`
// (residual added in its epilogue) followed by the LayerNorm kernel.  Two fusions were built and measured in rounds 1-2 (statistics +
// in-place pass inside the GEMM epilogue; "virtual" LayerNorm folded into the consumer GEMMs): both lost to this form on the
// power-capped board (65.1-67.1 k vs 68.0 k triplets/s) and were removed -- DESIGN.md section 5.
int gemm_layernorm(cir_ctx* ctx, const void* A, int64_t lda, int64_t a_bs, const void* W, int64_t ldw, int64_t w_bs, const float* bias,
                   int64_t bias_bs, const void* res, int64_t ldres, int64_t res_bs, const float* gamma, const float* beta, float eps,
                   void* pre, void* y, int64_t M, int64_t K, int batch) {
  const int64_t D_ = CIR_HIDDEN;
  CIR_TRY(gemm(ctx, A, lda, a_bs, W, ldw, w_bs, bias, bias_bs, pre, D_, M * D_, 0, res, ldres, res_bs, 0, M, D_, K, batch, CIR_ACT_NONE));
  return cir_add_layernorm(ctx, pre, 0, (int64_t)batch * M, nullptr, gamma, beta, M, y, 0, (int64_t)batch * M, eps);
}

constexpr int64_t D = CIR_HIDDEN, F = CIR_FFN;
constexpr float BERT_EPS = 1e-12f;   // configs/med_config.json:11
constexpr float VIT_EPS = 1e-6f;     // src/vit.py:142

}  // namespace

// ctx_s = softmax(Q K^T / 8 + mask) V of the text self-attention of `batch` streams (captions x L rows each, stream stride
// caps*L rows in hin / qkv / ctxout), Q|K|V = hin Wqkv^T + b.  bf16 with L in {8, 16, 24, 32}: one fused kernel (the projection never
// reaches HBM); otherwise the QKV GEMM into `qkv` followed by one attention call per stream.
static int self_attention(cir_ctx* ctx, const void* hin, const void* wqkv, const float* bqkv, int batch, const int32_t* mask,
                          const int32_t* mask_index, int64_t caps, int64_t L, void* qkv, void* ctxout) {
  const size_t es = act_size(ctx);
  const int64_t Mr = caps * L;
  if (ctx->fuse_qkv && cir_qkv_attention_supported(ctx, L)) {
    cir_qkv_attn_args q{};
    q.x = hin; q.x_bs = Mr * D; q.w = wqkv; q.bias = bqkv; q.out = ctxout; q.out_rs = D; q.out_bs = Mr * D;
    q.key_mask = mask; q.mask_index = mask_index; q.captions = caps; q.L = (int32_t)L; q.batch = batch; q.scale = 0.125f;
    return cir_qkv_attention(ctx, &q);
  }
  CIR_TRY(gemm(ctx, hin, D, Mr * D, wqkv, D, 3 * D * D, bqkv, 3 * D, qkv, 3 * D, Mr * 3 * D, 0, nullptr, 0, 0, 0, Mr, 3 * D, D, batch, CIR_ACT_NONE));
  for (int s = 0; s < batch; s++) {
    cir_attn_args a{};
    void* qkv_s = at(qkv, s * Mr * 3 * D, es);
    a.q = qkv_s; a.k = at(qkv_s, D, es); a.v = at(qkv_s, 2 * D, es); a.o = at(ctxout, s * Mr * D, es);
    a.q_bs = a.k_bs = a.v_bs = L * 3 * D; a.q_rs = a.k_rs = a.v_rs = 3 * D; a.o_bs = L * D; a.o_rs = D;
    a.key_mask = mask; a.mask_index = mask_index;
    a.B = (int32_t)caps; a.H = CIR_HEADS; a.Lq = (int32_t)L; a.Lk = (int32_t)L; a.scale = 0.125f;                   // / sqrt(64) (nlvr_encoder.py:193)
    CIR_TRY(cir_attention(ctx, &a));
  }
  return CIR_OK;
}

// self_attention for query row 0 (CLS) of each caption only; its keys/values still come from all L rows.  ctxout: [batch][caps]
// rows.  K | V for all rows (weight rows 768..2303 -> qkv columns 768..2303), Q for the CLS rows only (A row stride L*768 ->
// qkv row 0 of each caption).
static int self_attention_cls(cir_ctx* ctx, const void* hin, const void* wqkv, const float* bqkv, int batch, const int32_t* mask,
                              const int32_t* mask_index, int64_t caps, int64_t L, void* qkv, void* ctxout) {
  const size_t es = act_size(ctx);
  const int64_t Mr = caps * L;
  CIR_TRY(gemm(ctx, hin, D, Mr * D, at(const_cast<void*>(wqkv), D * D, es), D, 3 * D * D, bqkv + D, 3 * D,
               at(qkv, D, es), 3 * D, Mr * 3 * D, 0, nullptr, 0, 0, 0, Mr, 2 * D, D, batch, CIR_ACT_NONE));
  CIR_TRY(gemm(ctx, hin, L * D, Mr * D, wqkv, D, 3 * D * D, bqkv, 3 * D, qkv, L * 3 * D, Mr * 3 * D, 0,
               nullptr, 0, 0, 0, caps, D, D, batch, CIR_ACT_NONE));
  for (int s = 0; s < batch; s++) {
    cir_attn_args a{};
    void* qkv_s = at(qkv, s * Mr * 3 * D, es);
    a.q = qkv_s; a.k = at(qkv_s, D, es); a.v = at(qkv_s, 2 * D, es); a.o = at(ctxout, s * caps * D, es);
    a.q_bs = a.k_bs = a.v_bs = L * 3 * D; a.q_rs = a.k_rs = a.v_rs = 3 * D; a.o_bs = D; a.o_rs = D;
    a.key_mask = mask; a.mask_index = mask_index;
    a.B = (int32_t)caps; a.H = CIR_HEADS; a.Lq = 1; a.Lk = (int32_t)L; a.scale = 0.125f;
    CIR_TRY(cir_attention(ctx, &a));
  }
  return CIR_OK;
}

// ========================================================================================== ViT
struct VitWs { void *patches, *patch_out, *x, *y, *qkv, *ctx, *f; size_t total; };
static VitWs vit_plan(const cir_ctx* ctx, void* ws, size_t bytes, int64_t B, int64_t S) {
  const size_t es = act_size(ctx);
  const int64_t P = (S / 16) * (S / 16), N = P + 1;
  Bump b(ws, bytes);
  VitWs w;
  w.patches = b.take(B * P * D * es);
  w.patch_out = b.take(B * P * D * 4);
  w.x = b.take(B * N * D * 4);
  w.y = b.take(B * N * D * es);
  w.qkv = b.take(B * N * 3 * D * es);
  w.ctx = b.take(B * N * D * es);
  w.f = b.take(B * N * F * es);
  w.total = align_up(b.off, 256);
  return w;
}
extern "C" size_t cir_vit_workspace_bytes(const cir_ctx* ctx, int64_t B, int64_t image_size) {
  return vit_plan(ctx, nullptr, 0, B, image_size).total;
}

extern "C" int cir_vit_forward(cir_ctx* ctx, const cir_vit_weights* w, const float* images, int64_t B,
                               int64_t S, void* tokens, void* workspace, size_t workspace_bytes) {
  CIR_ENTER(ctx);
  if (B == 0) return CIR_OK;
  CIR_CHECK_ARG(S % 16 == 0 && S >= 16, "vit: image size %lld is not a multiple of 16", (long long)S);
  VitWs ws = vit_plan(ctx, workspace, workspace_bytes, B, S);
  if (workspace_bytes < ws.total) { cir_set_error("vit: workspace %zu < %zu", workspace_bytes, ws.total); return CIR_EWORKSPACE; }
  const int64_t P = (S / 16) * (S / 16), N = P + 1, R = B * N;
  // patch embedding: Conv2d(3,768,16,16) as im2col + GEMM (timm PatchEmbed; call site src/vit.py:144-145,182)
  CIR_TRY(cir_im2col16(ctx, images, ws.patches, B, (int)S));
  CIR_TRY(gemm(ctx, ws.patches, D, 0, w->patch_w, D, 0, w->patch_b, 0, ws.patch_out, D, 0, 1, nullptr, 0, 0, 0, B * P, D, D, 1, CIR_ACT_NONE));
  CIR_TRY(cir_vit_assemble(ctx, (const float*)ws.patch_out, w->cls_token, w->pos_embed, (float*)ws.x, B, N));   // :184-188
  for (int i = 0; i < CIR_LAYERS; i++) {                                                                           // :190-191
    // x = x + proj(attn(norm1(x)))   (src/vit.py:108, :70-86)
    CIR_TRY(cir_add_layernorm(ctx, ws.x, 1, R, nullptr, w->norm1_g[i], w->norm1_b[i], R, ws.y, 0, R, VIT_EPS));
    CIR_TRY(gemm(ctx, ws.y, D, 0, w->qkv_w[i], D, 0, w->qkv_b[i], 0, ws.qkv, 3 * D, 0, 0, nullptr, 0, 0, 0, R, 3 * D, D, 1, CIR_ACT_NONE));
    cir_attn_args a{};
    const size_t es = act_size(ctx);
    a.q = ws.qkv; a.k = at(ws.qkv, D, es); a.v = at(ws.qkv, 2 * D, es); a.o = ws.ctx;
    a.q_bs = a.k_bs = a.v_bs = N * 3 * D; a.q_rs = a.k_rs = a.v_rs = 3 * D;
    a.o_bs = N * D; a.o_rs = D;
    a.B = (int32_t)B; a.H = CIR_HEADS; a.Lq = (int32_t)N; a.Lk = (int32_t)N; a.scale = 0.125f;                   // head_dim ** -0.5 (:50)
    a.kv_batches = (int32_t)B;
    CIR_TRY(cir_attention(ctx, &a));
    CIR_TRY(gemm(ctx, ws.ctx, D, 0, w->proj_w[i], D, 0, w->proj_b[i], 0, ws.x, D, 0, 1, ws.x, D, 0, 1, R, D, D, 1, CIR_ACT_NONE));
    // x = x + fc2(gelu(fc1(norm2(x))))   (src/vit.py:109, :35-41)
    CIR_TRY(cir_add_layernorm(ctx, ws.x, 1, R, nullptr, w->norm2_g[i], w->norm2_b[i], R, ws.y, 0, R, VIT_EPS));
    CIR_TRY(gemm(ctx, ws.y, D, 0, w->fc1_w[i], D, 0, w->fc1_b[i], 0, ws.f, F, 0, 0, nullptr, 0, 0, 0, R, F, D, 1, CIR_ACT_GELU));
    CIR_TRY(gemm(ctx, ws.f, F, 0, w->fc2_w[i], F, 0, w->fc2_b[i], 0, ws.x, D, 0, 1, ws.x, D, 0, 1, R, D, F, 1, CIR_ACT_NONE));
  }
  CIR_TRY(cir_add_layernorm(ctx, ws.x, 1, R, nullptr, w->norm_g, w->norm_b, R, tokens, 0, R, VIT_EPS));          // :192
  return CIR_OK;
}

// ========================================================================================== stage I
struct S1Ws { void *reft, *h, *qkv, *ctx, *pre, *a, *qc, *kv, *x, *f, *cls; float* proj; size_t total; };
static S1Ws s1_plan(const cir_ctx* ctx, void* ws, size_t bytes, int64_t Q, int64_t L, int64_t N) {
  const size_t es = act_size(ctx);
  const int64_t R = Q * L;
  Bump b(ws, bytes);
  S1Ws w;
  w.reft = b.take(Q * N * D * es);
  w.h = b.take(R * D * es);
  w.qkv = b.take(R * 3 * D * es);
  w.ctx = b.take(R * D * es);
  w.pre = b.take(R * D * 4);
  w.a = b.take(R * D * es);
  w.qc = b.take(R * D * es);
  w.kv = b.take(Q * N * 2 * D * es);
  w.x = b.take(R * D * es);
  w.f = b.take(R * F * es);
  w.cls = b.take(Q * D * es);
  w.proj = (float*)b.take(Q * CIR_EMBED * 4);
  w.total = align_up(b.off, 256);
  return w;
}
extern "C" size_t cir_stage1_workspace_bytes(const cir_ctx* ctx, int64_t Q, int64_t L, int64_t N) {
  return s1_plan(ctx, nullptr, 0, Q, L, N).total;
}

static int project_normalize(cir_ctx* ctx, const void* cls_rows, int64_t lda, const void* W, const float* bias, int64_t rows,
                             float* tmp, float* out, int twice) {
  CIR_TRY(gemm(ctx, cls_rows, lda, 0, W, D, 0, bias, 0, tmp, CIR_EMBED, 0, 1, nullptr, 0, 0, 0, rows, CIR_EMBED, D, 1, CIR_ACT_NONE));
  CIR_TRY(cir_l2_normalize(ctx, tmp, out, rows, CIR_EMBED));
  if (twice) CIR_TRY(cir_l2_normalize(ctx, out, out, rows, CIR_EMBED));
  return CIR_OK;
}

extern "C" int cir_stage1_encode(cir_ctx* ctx, const cir_stage1_weights* w, const void* gallery_tokens,
                                 const int32_t* ref_index, const int32_t* ids, const int32_t* mask,
                                 int64_t Q, int64_t L, int64_t N, void* z_t, float* q_emb, int normalize_twice,
                                 void* workspace, size_t workspace_bytes) {
  CIR_ENTER(ctx);
  if (Q == 0) return CIR_OK;
  CIR_CHECK_ARG(L >= 1 && L <= 512 && N >= 1 && N <= 1024, "stage1: L=%lld N=%lld out of range", (long long)L, (long long)N);
  S1Ws ws = s1_plan(ctx, workspace, workspace_bytes, Q, L, N);
  if (workspace_bytes < ws.total) { cir_set_error("stage1: workspace %zu < %zu", workspace_bytes, ws.total); return CIR_EWORKSPACE; }
  const size_t es = act_size(ctx);
  const int64_t R = Q * L;
  CIR_TRY(cir_gather_rows(ctx, gallery_tokens, ref_index, ws.reft, Q, N * D));
  CIR_TRY(cir_bert_embeddings(ctx, ids, Q, L, w->word_emb, w->pos_emb, w->emb_ln_g, w->emb_ln_b, ws.h));         // med.py:86-110
  for (int i = 0; i < CIR_LAYERS; i++) {                                                                           // med.py:348-398
    CIR_TRY(self_attention(ctx, ws.h, w->self_qkv_w[i], w->self_qkv_b[i], 1, mask, nullptr, Q, L, ws.qkv, ws.ctx));   // med.py:112-216
    CIR_TRY(gemm(ctx, ws.ctx, D, 0, w->self_out_w[i], D, 0, w->self_out_b[i], 0, ws.pre, D, 0, 0, ws.h, D, 0, 0, R, D, D, 1, CIR_ACT_NONE));
    CIR_TRY(cir_add_layernorm(ctx, ws.pre, 0, R, nullptr, w->self_ln_g[i], w->self_ln_b[i], R, ws.a, 0, R, BERT_EPS));
    // cross-attention onto the reference image tokens (all-ones encoder mask -> +0)
    CIR_TRY(gemm(ctx, ws.a, D, 0, w->cross_q_w[i], D, 0, w->cross_q_b[i], 0, ws.qc, D, 0, 0, nullptr, 0, 0, 0, R, D, D, 1, CIR_ACT_NONE));
    CIR_TRY(gemm(ctx, ws.reft, D, 0, w->cross_kv_w[i], D, 0, w->cross_kv_b[i], 0, ws.kv, 2 * D, 0, 0, nullptr, 0, 0, 0, Q * N, 2 * D, D, 1, CIR_ACT_NONE));
    cir_attn_args c{};
    c.q = ws.qc; c.k = ws.kv; c.v = at(ws.kv, D, es); c.o = ws.ctx;
    c.q_bs = L * D; c.q_rs = D; c.k_bs = c.v_bs = N * 2 * D; c.k_rs = c.v_rs = 2 * D; c.o_bs = L * D; c.o_rs = D;
    c.B = (int32_t)Q; c.H = CIR_HEADS; c.Lq = (int32_t)L; c.Lk = (int32_t)N; c.scale = 0.125f;
    c.kv_batches = (int32_t)Q;
    CIR_TRY(cir_attention(ctx, &c));
    CIR_TRY(gemm(ctx, ws.ctx, D, 0, w->cross_out_w[i], D, 0, w->cross_out_b[i], 0, ws.pre, D, 0, 0, ws.a, D, 0, 0, R, D, D, 1, CIR_ACT_NONE));
    CIR_TRY(cir_add_layernorm(ctx, ws.pre, 0, R, nullptr, w->cross_ln_g[i], w->cross_ln_b[i], R, ws.x, 0, R, BERT_EPS));
    CIR_TRY(gemm(ctx, ws.x, D, 0, w->ffn1_w[i], D, 0, w->ffn1_b[i], 0, ws.f, F, 0, 0, nullptr, 0, 0, 0, R, F, D, 1, CIR_ACT_GELU));
    CIR_TRY(gemm(ctx, ws.f, F, 0, w->ffn2_w[i], F, 0, w->ffn2_b[i], 0, ws.pre, D, 0, 0, ws.x, D, 0, 0, R, D, F, 1, CIR_ACT_NONE));
    CIR_TRY(cir_add_layernorm(ctx, ws.pre, 0, R, nullptr, w->ffn_ln_g[i], w->ffn_ln_b[i], R, ws.h, 0, R, BERT_EPS));
  }
  if (z_t) CIR_TRY(cir_gather_rows(ctx, ws.h, nullptr, z_t, R, D));                                               // return_raw=True
  if (q_emb) CIR_TRY(project_normalize(ctx, ws.h, L * D, w->text_proj_w, w->text_proj_b, Q, ws.proj, q_emb, normalize_twice));  // blip_stage1.py:83
  return CIR_OK;
}

extern "C" int cir_stage1_gallery_embed(cir_ctx* ctx, const cir_stage1_weights* w, const void* tokens, int64_t G,
                                        int64_t N, float* g_emb, void* workspace, size_t workspace_bytes) {
  CIR_ENTER(ctx);
  if (G == 0) return CIR_OK;
  const size_t need = align_up((size_t)G * CIR_EMBED * 4, 256);
  if (workspace_bytes < need) { cir_set_error("gallery_embed: workspace %zu < %zu", workspace_bytes, need); return CIR_EWORKSPACE; }
  return project_normalize(ctx, tokens, N * D, w->vision_proj_w, w->vision_proj_b, G, (float*)workspace, g_emb, 0);   // blip_stage1.py:57
}

// ========================================================================================== stage II
// Where a stage-II call's cross-attention K/V come from:
//   KV_PROJECT      the chunk's candidate tokens, gathered and projected per layer into the workspace
//   KV_CACHE        a bf16 / fp32 cir_stage2_kv_cache, read in place: one int32 cache row per triplet in the workspace
//   KV_CACHE_MXFP8  an MXFP8 cache: the K/V of the C candidates dequantised per layer into the workspace (the KV_PROJECT layout)
enum KvSrc { KV_PROJECT, KV_CACHE, KV_CACHE_MXFP8 };
static KvSrc kv_src(const cir_stage2_kv_cache* c) { return !c ? KV_PROJECT : c->dtype == CIR_KV_MXFP8 ? KV_CACHE_MXFP8 : KV_CACHE; }
// a cache of the context's dtype, or an MXFP8 cache in a bf16 context
static bool kv_cache_serves(const cir_ctx* ctx, const cir_stage2_kv_cache* c) {
  return c->dtype == ctx->dtype || (c->dtype == CIR_KV_MXFP8 && ctx->dtype == CIR_DTYPE_BF16);
}

struct S2Ws { void *cand, *kv, *emb, *h, *qkv, *ctx, *pre, *a, *qc, *ctxc, *m, *x, *f, *feats; float *hid; int32_t* kv_row; size_t total; };
static S2Ws s2_plan(const cir_ctx* ctx, void* ws, size_t bytes, int64_t T, int64_t C, int64_t Q, int64_t L, int64_t N, KvSrc src = KV_PROJECT) {
  const size_t es = act_size(ctx);
  const int64_t M = T * L;
  Bump b(ws, bytes);
  S2Ws w;
  w.cand = src == KV_PROJECT ? b.take(C * N * D * es) : nullptr;
  w.kv = src == KV_CACHE ? nullptr : b.take(C * N * 4 * D * es);
  w.emb = b.take(Q * L * D * es);
  w.h = b.take(2 * M * D * es);
  w.qkv = b.take(2 * M * 3 * D * es);
  w.ctx = b.take(2 * M * D * es);
  w.pre = b.take(2 * M * D * 4);
  w.a = b.take(2 * M * D * es);
  w.qc = b.take(2 * M * D * es);
  w.ctxc = b.take(M * 2 * D * es);
  w.m = b.take(M * D * 4);
  w.x = b.take(2 * M * D * es);
  w.f = b.take(2 * M * F * es);
  w.feats = b.take(T * 2 * D * es);
  w.hid = (float*)b.take(T * D * 4);
  w.kv_row = src == KV_CACHE ? (int32_t*)b.take(T * 4) : nullptr;
  w.total = align_up(b.off, 256);
  return w;
}
extern "C" size_t cir_stage2_workspace_bytes(const cir_ctx* ctx, int64_t T, int64_t C, int64_t Q, int64_t L, int64_t N) {
  return s2_plan(ctx, nullptr, 0, T, C, Q, L, N).total;
}

// Layer 0's query-only part (both streams): QKV, masked self-attention, dense + LayerNorm{A,B} -> a_out, cross query
// projection -> qc_out, for Q queries whose layer inputs sit in hq = [2][Q*L][768] (stream 0 = z_t, stream 1 =
// embeddings).  qkv / ctxbuf / scratch: [2][Q*L][2304 / 768 / 768] temporaries; a_out / qc_out: [2][Q*L][768].
static int stage2_query_block(cir_ctx* ctx, const cir_stage2_weights* w, const void* hq, const int32_t* mask, int64_t Q, int64_t L,
                              void* qkv, void* ctxbuf, void* scratch, void* a_out, void* qc_out) {
  const size_t es = act_size(ctx);
  const int64_t Mq = Q * L;
  CIR_TRY(self_attention(ctx, hq, w->self_qkv_w[0], w->self_qkv_b[0], 2, mask, nullptr, Q, L, qkv, ctxbuf));   // mask row q belongs to query q
  CIR_TRY(gemm_layernorm(ctx, ctxbuf, D, Mq * D, w->self_out_w[0], D, D * D, w->self_out_b[0], D, hq, D, Mq * D,
                         w->self_ln_g[0], w->self_ln_b[0], BERT_EPS, scratch, a_out, Mq, D, 2));
  return gemm(ctx, a_out, D, Mq * D, w->cross_q_w[0], D, D * D, w->cross_q_b[0], D, qc_out, D, Mq * D, 0, nullptr, 0, 0, 0,
              Mq, D, D, 2, CIR_ACT_NONE);
}

// stream 0 = z_t WITHOUT embedding LayerNorm (nlvr_encoder.py:892), stream 1 = embeddings (:880-886), for Q queries
static int stage2_query_inputs(cir_ctx* ctx, const cir_stage2_weights* w, const void* z_t, const int32_t* ids, int64_t Q, int64_t L, void* hq) {
  CIR_TRY(cir_gather_rows(ctx, z_t, nullptr, hq, Q, L * D));
  return cir_bert_embeddings(ctx, ids, Q, L, w->word_emb, w->pos_emb, w->emb_ln_g, w->emb_ln_b, at(hq, Q * L * D, act_size(ctx)));
}

struct S2PrefixWs { void *hq, *qkv, *ctx, *scratch; size_t total; };
static S2PrefixWs s2_prefix_plan(const cir_ctx* ctx, void* ws, size_t bytes, int64_t Q, int64_t L) {
  const size_t es = act_size(ctx);
  const int64_t Mq = Q * L;
  Bump b(ws, bytes);
  S2PrefixWs w;
  w.hq = b.take(2 * Mq * D * es);
  w.qkv = b.take(2 * Mq * 3 * D * es);
  w.ctx = b.take(2 * Mq * D * es);
  w.scratch = b.take(2 * Mq * D * 4);
  w.total = align_up(b.off, 256);
  return w;
}
extern "C" size_t cir_stage2_prefix_workspace_bytes(const cir_ctx* ctx, int64_t Q, int64_t L) { return s2_prefix_plan(ctx, nullptr, 0, Q, L).total; }

extern "C" int cir_stage2_prefix(cir_ctx* ctx, const cir_stage2_weights* w, const void* z_t, const int32_t* ids, const int32_t* mask,
                                 int64_t Q, int64_t L, void* a0, void* qc0, void* workspace, size_t workspace_bytes) {
  CIR_ENTER(ctx);
  if (Q == 0) return CIR_OK;
  CIR_CHECK_ARG(L >= 1 && L <= 512 && z_t && ids && mask && a0 && qc0, "stage2_prefix: bad argument");
  S2PrefixWs ws = s2_prefix_plan(ctx, workspace, workspace_bytes, Q, L);
  if (workspace_bytes < ws.total) { cir_set_error("stage2_prefix: workspace %zu < %zu", workspace_bytes, ws.total); return CIR_EWORKSPACE; }
  CIR_TRY(stage2_query_inputs(ctx, w, z_t, ids, Q, L, ws.hq));
  return stage2_query_block(ctx, w, ws.hq, mask, Q, L, ws.qkv, ws.ctx, ws.scratch, a0, qc0);
}

// kv_row[t] = cand_list[trip_slot[t]] - row0: the cache row of each triplet's candidate (the attention's kv_index)
__global__ void stage2_kv_rows_kernel(const int32_t* __restrict__ cand_list, const int32_t* __restrict__ trip_slot, int64_t row0,
                                      int64_t T, int32_t* __restrict__ kv_row) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < T) kv_row[t] = (int32_t)(cand_list[trip_slot[t]] - row0);
}

// K/V rows of layer i in a cache: act [rows * N][4 * 768]
static const void* kv_cache_layer(const cir_stage2_kv_cache* c, int i, size_t es) {
  return (const char*)c->kv + (int64_t)i * c->rows * c->num_tokens * 4 * D * (int64_t)es;
}

// cache == NULL: the chunk's candidate tokens are gathered and their K/V projected per layer into the workspace (attention reads
// K/V batch trip_slot[t] of C); a bf16 / fp32 cache: the K/V rows come from the cache (K/V batch kv_row[t] of cache->rows); an
// MXFP8 cache: the K/V of the C candidates are dequantised per layer into the workspace (K/V batch trip_slot[t] of C).
// tile_counts (cached only; NULL from every host-planned caller): device {tiles, cls tiles} of an on-device plan
// (cir_stage2_plan_topk).  attn_tiles / attn_tiles_cls then hold at most T entries, of which the two cross-attentions read as many
// as the device counts say, and trip_slot holds each triplet's cache row -- or, with an MXFP8 cache, its run number, cand_list the
// runs' gallery rows and cand_count (device) how many of the C entries the plan filled.
static int stage2_score_impl(cir_ctx* ctx, const cir_stage2_weights* w, const void* gallery_tokens,
                             const int32_t* cand_list, int64_t C, const void* z_t, const int32_t* ids,
                             const int32_t* mask, int64_t Q, int64_t L, int64_t N,
                             const int32_t* trip_query, const int32_t* trip_slot, int64_t T,
                             const int32_t* attn_work, int64_t num_attn_work,
                             const int32_t* attn_tiles, int64_t num_attn_tiles,
                             const int32_t* attn_tiles_cls, int64_t num_attn_tiles_cls,
                             float* scores, float* feats, void* workspace, size_t workspace_bytes,
                             const void* a0, const void* qc0,              // optional cir_stage2_prefix results of the Q queries
                             const cir_stage2_kv_cache* cache, const int32_t* tile_counts = nullptr,
                             const int32_t* cand_count = nullptr) {
  if (T == 0) return CIR_OK;
  CIR_CHECK_ARG(C >= 1 && Q >= 1, "stage2: need at least one candidate and one query");
  CIR_CHECK_ARG(L >= 1 && L <= 512 && N >= 1 && N <= 1024, "stage2: L=%lld N=%lld out of range", (long long)L, (long long)N);
  const KvSrc src = kv_src(cache);
  S2Ws ws = s2_plan(ctx, workspace, workspace_bytes, T, C, Q, L, N, src);
  if (workspace_bytes < ws.total) { cir_set_error("stage2: workspace %zu < %zu", workspace_bytes, ws.total); return CIR_EWORKSPACE; }
  const size_t es = act_size(ctx);
  const int64_t M = T * L;
  const int32_t* kv_index = trip_slot;
  int32_t kv_batches = (int32_t)C;
  if (src == KV_CACHE && tile_counts) {
    kv_batches = (int32_t)cache->rows;               // trip_slot already holds the cache rows
  } else if (src == KV_CACHE) {
    stage2_kv_rows_kernel<<<(unsigned)((T + 255) / 256), 256, 0, ctx->stream>>>(cand_list, trip_slot, cache->row0, T, ws.kv_row);
    CIR_LAUNCH_CHECK(ctx);
    kv_index = ws.kv_row;
    kv_batches = (int32_t)cache->rows;
  } else if (src == KV_PROJECT) {
    // candidate tokens of this chunk, contiguous [C*N, 768] (validate_stage2.py:251 gather, once per unique image)
    CIR_TRY(cir_gather_rows(ctx, gallery_tokens, cand_list, ws.cand, C, N * D));
  }
  // stream 1 = embeddings (nlvr_encoder.py:880-886), stream 0 = z_t WITHOUT embedding LayerNorm (:892);
  // both expanded over the query's triplets (blip_stage2.py:118-124)
  // The inputs of layer 0 -- and with them its whole self-attention block and its cross-attention query projection --
  // depend on the QUERY only, not on the candidate (both streams are expanded copies, blip_stage2.py:118-124): run them
  // once per unique query of the chunk ([2][Q*L] rows) and expand the results over the triplets.  Exact.
  static_assert(CIR_LAYERS >= 2, "layer 0 is never the CLS-only last layer");
  const bool prefixed = a0 != nullptr;
  CIR_CHECK_ARG(!prefixed || qc0, "stage2: a0 and qc0 come as a pair");
  const bool dedup0 = prefixed || (ctx->dedup_first && Q <= T);
  const int64_t Mq = Q * L;
  // layer 0's a / qc rows of the Q queries, [2][Q*L] rows each: precomputed for the whole query set (cir_stage2_prefix) or
  // computed here once per unique query (stage2_query_block)
  const void* a_q = a0;
  const void* q_q = qc0;
  if (prefixed) {
    // nothing to prepare: layer 0 starts from the expanded a0 / qc0 rows
  } else if (dedup0) {
    CIR_TRY(stage2_query_inputs(ctx, w, z_t, ids, Q, L, ws.h));
    // a_q -> ws.pre, its pre-LayerNorm scratch -> ws.x, q_q -> ws.qkv (written after the self-attention has read the
    // QKV rows); all are [2][Q*L] rows and Q <= T, so the [2][T*L]-row buffers hold them
    CIR_TRY(stage2_query_block(ctx, w, ws.h, mask, Q, L, ws.qkv, ws.ctx, ws.x, ws.pre, ws.qkv));
    a_q = ws.pre; q_q = ws.qkv;
  } else {
    CIR_TRY(cir_bert_embeddings(ctx, ids, Q, L, w->word_emb, w->pos_emb, w->emb_ln_g, w->emb_ln_b, ws.emb));
    CIR_TRY(cir_gather_rows(ctx, z_t, trip_query, ws.h, T, L * D));
    CIR_TRY(cir_gather_rows(ctx, ws.emb, trip_query, at(ws.h, M * D, es), T, L * D));
  }
  // ---- layer i from its cross-attention on: twin cross-attention onto the SAME candidate tokens (:322-339), merge, FFN, over the
  // [2][T*Lq] rows of ws.a / ws.qc (Lq query rows per triplet) into ws.h.  tiles / work / counts: the cross-attention's tile list,
  // work list and device tile count for Lq-row queries.
  auto cross_ffn = [&](int i, int64_t Lq, const int32_t* tiles, int64_t num_tiles, const int32_t* work, int64_t num_work,
                       const int32_t* counts) -> int {
    const int64_t R = T * Lq;
    // K/V projections once per candidate image: rows K0|V0|K1|V1 (:158-159)
    void* kv = src == KV_CACHE ? const_cast<void*>(kv_cache_layer(cache, i, es)) : ws.kv;
    if (src == KV_PROJECT)
      CIR_TRY(gemm(ctx, ws.cand, D, 0, w->cross_kv_w[i], D, 0, w->cross_kv_b[i], 0, ws.kv, 4 * D, 0, 0, nullptr, 0, 0, 0,
                   C * N, 4 * D, D, 1, CIR_ACT_NONE));
    else if (src == KV_CACHE_MXFP8)
      CIR_TRY(cir_kv_mxfp8_dequant(ctx, cache, i, cand_list, C, cand_count, ws.kv));
    for (int s = 0; s < 2; s++) {
      cir_attn_args c{};
      c.q = at(ws.qc, s * R * D, es); c.k = at(kv, s * 2 * D, es); c.v = at(kv, s * 2 * D + D, es);
      c.o = at(ws.ctxc, s * D, es);
      c.q_bs = Lq * D; c.q_rs = D; c.k_bs = c.v_bs = N * 4 * D; c.k_rs = c.v_rs = 4 * D; c.o_bs = Lq * 2 * D; c.o_rs = 2 * D;
      c.kv_index = kv_index;
      c.work = work; c.num_work = (int32_t)num_work;
      c.tiles = tiles; c.num_tiles = (int32_t)num_tiles; c.kv_batches = kv_batches;
      c.B = (int32_t)T; c.H = CIR_HEADS; c.Lq = (int32_t)Lq; c.Lk = (int32_t)N; c.scale = 0.125f;
      CIR_TRY(counts ? cir_attention_counted(ctx, &c, counts) : cir_attention(ctx, &c));
    }
    // m = merge(dense0(c0), dense1(c1)) folded into one K=1536 GEMM (:250-258); x_s = LayerNorm{A,B}(m + a_s) (:256,:260)
    CIR_TRY(gemm(ctx, ws.ctxc, 2 * D, 0, w->cross_out_w[i], 2 * D, 0, w->cross_out_b[i], 0, ws.m, D, 0, 0, nullptr, 0, 0, 0,
                 R, D, 2 * D, 1, CIR_ACT_NONE));
    CIR_TRY(cir_add_layernorm(ctx, ws.m, 0, R, ws.a, w->cross_ln_g[i], w->cross_ln_b[i], R, ws.x, 0, 2 * R, BERT_EPS));
    // ---- FFN, weights shared by both streams (:469-476): both streams as 2R rows
    CIR_TRY(gemm(ctx, ws.x, D, 0, w->ffn1_w[i], D, 0, w->ffn1_b[i], 0, ws.f, F, 0, 0, nullptr, 0, 0, 0, 2 * R, F, D, 1, CIR_ACT_GELU));
    return gemm_layernorm(ctx, ws.f, F, 0, w->ffn2_w[i], F, 0, w->ffn2_b[i], 0, ws.x, D, 0, w->ffn_ln_g[i], w->ffn_ln_b[i], BERT_EPS,
                          ws.pre, ws.h, 2 * R, F, 1);
  };
  for (int i = 0; i < CIR_LAYERS; i++) {                                                                           // nlvr_encoder.py:506
    // With prune_last, layer 11 runs on the CLS rows only: the encoder returns cat(h0[:,0,:], h1[:,0,:]) (nlvr_encoder.py:906-909),
    // so there only query row 0 of each stream feeds the result; its keys/values still come from all L rows (self) and all N image
    // tokens (cross).
    const bool cls = ctx->prune_last && i == CIR_LAYERS - 1;
    const int64_t Lq = cls ? 1 : L, R = T * Lq;
    if (dedup0 && i == 0) {
      for (int s = 0; s < 2; s++) {                           // expand over the triplets (blip_stage2.py:118-124)
        CIR_TRY(cir_gather_rows(ctx, at(const_cast<void*>(a_q), s * Mq * D, es), trip_query, at(ws.a, s * M * D, es), T, L * D));
        CIR_TRY(cir_gather_rows(ctx, at(const_cast<void*>(q_q), s * Mq * D, es), trip_query, at(ws.qc, s * M * D, es), T, L * D));
      }
    } else {
      // ---- twin self-attention (:281-289, :346-363): separate weights per stream, shared padding mask (:774)
      if (cls)
        CIR_TRY(self_attention_cls(ctx, ws.h, w->self_qkv_w[i], w->self_qkv_b[i], 2, mask, trip_query, T, L, ws.qkv, ws.ctx));
      else
        CIR_TRY(self_attention(ctx, ws.h, w->self_qkv_w[i], w->self_qkv_b[i], 2, mask, trip_query, T, L, ws.qkv, ws.ctx));
      // a_s = LayerNorm{A,B}(dense_s(ctx_s) + h_s)   (:261-264)
      CIR_TRY(gemm_layernorm(ctx, ws.ctx, D, R * D, w->self_out_w[i], D, D * D, w->self_out_b[i], D, ws.h, cls ? L * D : D, M * D,
                             w->self_ln_g[i], w->self_ln_b[i], BERT_EPS, ws.pre, ws.a, R, D, 2));
      CIR_TRY(gemm(ctx, ws.a, D, R * D, w->cross_q_w[i], D, D * D, w->cross_q_b[i], D, ws.qc, D, R * D, 0, nullptr, 0, 0, 0,
                   R, D, D, 2, CIR_ACT_NONE));
    }
    // the mma.sync work list describes L-row units: the CLS layer gets none
    if (cls)
      CIR_TRY(cross_ffn(i, Lq, attn_tiles_cls, num_attn_tiles_cls, nullptr, 0, tile_counts ? tile_counts + 1 : nullptr));
    else
      CIR_TRY(cross_ffn(i, Lq, attn_tiles, num_attn_tiles, attn_work, num_attn_work, tile_counts));
  }
  // cat(CLS0, CLS1) (:909) -> cls_head (blip_stage2.py:50-54,134-136)
  CIR_TRY(cir_gather_cls(ctx, ws.h, T, ctx->prune_last ? 1 : L, ws.feats, feats));
  CIR_TRY(gemm(ctx, ws.feats, 2 * D, 0, w->cls0_w, 2 * D, 0, w->cls0_b, 0, ws.hid, D, 0, 1, nullptr, 0, 0, 0, T, D, 2 * D, 1, CIR_ACT_RELU));
  CIR_TRY(cir_head_dot(ctx, ws.hid, w->cls2_w, w->cls2_b, scores, T));
  return CIR_OK;
}

extern "C" int cir_stage2_score(cir_ctx* ctx, const cir_stage2_weights* w, const void* gallery_tokens,
                                const int32_t* cand_list, int64_t C, const void* z_t, const int32_t* ids,
                                const int32_t* mask, int64_t Q, int64_t L, int64_t N,
                                const int32_t* trip_query, const int32_t* trip_slot, int64_t T,
                                const int32_t* attn_work, int64_t num_attn_work,
                                const int32_t* attn_tiles, int64_t num_attn_tiles,
                                const int32_t* attn_tiles_cls, int64_t num_attn_tiles_cls,
                                float* scores, float* feats, void* workspace, size_t workspace_bytes) {
  CIR_ENTER(ctx);
  CIR_CHECK_ARG(T == 0 || (z_t && ids), "stage2: z_t and ids are required");
  return stage2_score_impl(ctx, w, gallery_tokens, cand_list, C, z_t, ids, mask, Q, L, N, trip_query, trip_slot, T, attn_work, num_attn_work,
                           attn_tiles, num_attn_tiles, attn_tiles_cls, num_attn_tiles_cls, scores, feats, workspace, workspace_bytes,
                           nullptr, nullptr, nullptr);
}

extern "C" int cir_stage2_score_prefixed(cir_ctx* ctx, const cir_stage2_weights* w, const void* gallery_tokens,
                                         const int32_t* cand_list, int64_t C, const void* a0, const void* qc0,
                                         const int32_t* mask, int64_t Q, int64_t L, int64_t N,
                                         const int32_t* trip_query, const int32_t* trip_slot, int64_t T,
                                         const int32_t* attn_work, int64_t num_attn_work,
                                         const int32_t* attn_tiles, int64_t num_attn_tiles,
                                         const int32_t* attn_tiles_cls, int64_t num_attn_tiles_cls,
                                         float* scores, float* feats, void* workspace, size_t workspace_bytes) {
  CIR_ENTER(ctx);
  CIR_CHECK_ARG(T == 0 || (a0 && qc0), "stage2_score_prefixed: a0 and qc0 are required");
  return stage2_score_impl(ctx, w, gallery_tokens, cand_list, C, nullptr, nullptr, mask, Q, L, N, trip_query, trip_slot, T, attn_work,
                           num_attn_work, attn_tiles, num_attn_tiles, attn_tiles_cls, num_attn_tiles_cls, scores, feats, workspace,
                           workspace_bytes, a0, qc0, nullptr);
}

// ------------------------------------------------------------------------------------------ resident K/V gallery
extern "C" size_t cir_stage2_kv_cache_bytes(const cir_ctx* ctx, int64_t rows, int64_t N) {
  if (rows < 0 || N < 0) return 0;
  return align_up((size_t)CIR_LAYERS * rows * N * 4 * D * act_size(ctx), 256);
}

// MXFP8: one e4m3 byte per element plus one E8M0 byte per 32 elements
extern "C" size_t cir_stage2_kv_cache_bytes_mxfp8(const cir_ctx*, int64_t rows, int64_t N) {
  if (rows < 0 || N < 0) return 0;
  return align_up((size_t)CIR_LAYERS * rows * N * (4 * D + 4 * D / 32), 256);
}

// the checks and record of _init / _init_mxfp8; `need` is the blob size of the cache format `fmt`
static int kv_cache_init(const char* what, void* blob, size_t bytes, int64_t row0, int64_t rows, int64_t N, size_t need, int fmt,
                         cir_stage2_kv_cache* out) {
  CIR_CHECK_ARG(out != nullptr, "%s: out is NULL", what);
  CIR_CHECK_ARG(row0 >= 0 && rows >= 0 && row0 + rows <= (1ll << 31) && N >= 1 && N <= 1024,
                "%s: bad range row0=%lld rows=%lld N=%lld", what, (long long)row0, (long long)rows, (long long)N);
  CIR_CHECK_ARG(rows * N < (1ll << 31), "%s: rows * N must stay below 2^31 (attention row index)", what);
  CIR_CHECK_ARG(rows == 0 || (blob && ((uintptr_t)blob & 255) == 0), "%s: blob must be 256-byte aligned", what);
  CIR_CHECK_ARG(bytes >= need, "%s: blob %zu < %zu bytes", what, bytes, need);
  out->row0 = row0; out->rows = rows; out->num_tokens = N; out->dtype = fmt; out->kv = blob;
  return CIR_OK;
}

extern "C" int cir_stage2_kv_cache_init(cir_ctx* ctx, void* blob, size_t bytes, int64_t row0, int64_t rows, int64_t N,
                                        cir_stage2_kv_cache* out) {
  return kv_cache_init("stage2_kv_cache_init", blob, bytes, row0, rows, N, cir_stage2_kv_cache_bytes(ctx, rows, N), ctx->dtype, out);
}

extern "C" int cir_stage2_kv_cache_init_mxfp8(cir_ctx* ctx, void* blob, size_t bytes, int64_t row0, int64_t rows, int64_t N,
                                              cir_stage2_kv_cache* out) {
  CIR_CHECK_ARG(ctx->dtype == CIR_DTYPE_BF16, "stage2_kv_cache_init_mxfp8: an MXFP8 cache needs a bf16 context (dtype %d)", ctx->dtype);
  return kv_cache_init("stage2_kv_cache_init_mxfp8", blob, bytes, row0, rows, N, cir_stage2_kv_cache_bytes_mxfp8(ctx, rows, N),
                       CIR_KV_MXFP8, out);
}

extern "C" int cir_stage2_kv_cache_fill(cir_ctx* ctx, const cir_stage2_weights* w, cir_stage2_kv_cache* cache, const void* tokens,
                                        int64_t first, int64_t n) {
  CIR_ENTER(ctx);
  CIR_CHECK_ARG(w && cache, "stage2_kv_cache_fill: NULL weights or cache");
  CIR_CHECK_ARG(cache->dtype == ctx->dtype, "stage2_kv_cache_fill: cache dtype %d, context dtype %d", cache->dtype, ctx->dtype);
  CIR_CHECK_ARG(n >= 0 && first >= cache->row0 && first + n <= cache->row0 + cache->rows,
                "stage2_kv_cache_fill: rows [%lld, %lld) outside the cache's [%lld, %lld)", (long long)first, (long long)(first + n),
                (long long)cache->row0, (long long)(cache->row0 + cache->rows));
  if (n == 0) return CIR_OK;
  CIR_CHECK_ARG(tokens != nullptr, "stage2_kv_cache_fill: tokens is NULL");
  const size_t es = act_size(ctx);
  const int64_t N = cache->num_tokens;
  // the pair tile whatever n is: a row's bytes must not depend on how many rows share its call
  ctx->gemm_force_pair = 1;
  int rc = CIR_OK;
  for (int i = 0; i < CIR_LAYERS && rc == CIR_OK; i++) {
    void* dst = at(const_cast<void*>(kv_cache_layer(cache, i, es)), (first - cache->row0) * N * 4 * D, es);
    rc = gemm(ctx, tokens, D, 0, w->cross_kv_w[i], D, 0, w->cross_kv_b[i], 0, dst, 4 * D, 0, 0, nullptr, 0, 0, 0, n * N, 4 * D, D, 1,
              CIR_ACT_NONE);
  }
  ctx->gemm_force_pair = 0;
  return rc;
}

extern "C" size_t cir_stage2_kv_cache_fill_mxfp8_workspace_bytes(const cir_ctx*, const cir_stage2_kv_cache* cache, int64_t slice_rows) {
  if (!cache || slice_rows < 0) return 0;
  return align_up((size_t)slice_rows * cache->num_tokens * 4 * D * sizeof(bf16), 256);
}

extern "C" int cir_stage2_kv_cache_fill_mxfp8(cir_ctx* ctx, const cir_stage2_weights* w, cir_stage2_kv_cache* cache, const void* tokens,
                                              int64_t first, int64_t n, void* workspace, size_t workspace_bytes) {
  CIR_ENTER(ctx);
  CIR_CHECK_ARG(w && cache, "stage2_kv_cache_fill_mxfp8: NULL weights or cache");
  CIR_CHECK_ARG(cache->dtype == CIR_KV_MXFP8 && ctx->dtype == CIR_DTYPE_BF16,
                "stage2_kv_cache_fill_mxfp8: cache format %d, context dtype %d (needs an MXFP8 cache and a bf16 context)", cache->dtype,
                ctx->dtype);
  CIR_CHECK_ARG(n >= 0 && first >= cache->row0 && first + n <= cache->row0 + cache->rows,
                "stage2_kv_cache_fill_mxfp8: rows [%lld, %lld) outside the cache's [%lld, %lld)", (long long)first,
                (long long)(first + n), (long long)cache->row0, (long long)(cache->row0 + cache->rows));
  if (n == 0) return CIR_OK;
  CIR_CHECK_ARG(tokens != nullptr, "stage2_kv_cache_fill_mxfp8: tokens is NULL");
  const int64_t N = cache->num_tokens, rn = cache->rows * N;
  const size_t row_bytes = (size_t)N * 4 * D * sizeof(bf16);
  const int64_t slice = workspace ? std::min<int64_t>(n, (int64_t)(workspace_bytes / row_bytes)) : 0;
  if (slice < 1) {
    cir_set_error("stage2_kv_cache_fill_mxfp8: workspace %zu < %zu (one row)", workspace ? workspace_bytes : 0, row_bytes);
    return CIR_EWORKSPACE;
  }
  uint8_t* elems = (uint8_t*)cache->kv;
  uint8_t* scales = elems + CIR_LAYERS * rn * 4 * D;
  // per slice and layer: the bf16 K/V of _fill (the pair tile whatever the slice is) into the workspace, then quantised
  ctx->gemm_force_pair = 1;
  int rc = CIR_OK;
  for (int64_t s0 = 0; s0 < n && rc == CIR_OK; s0 += slice) {
    const int64_t m = std::min(slice, n - s0), r = (first - cache->row0 + s0) * N;
    const void* tok = at(const_cast<void*>(tokens), s0 * N * D, sizeof(bf16));
    for (int i = 0; i < CIR_LAYERS && rc == CIR_OK; i++) {
      rc = gemm(ctx, tok, D, 0, w->cross_kv_w[i], D, 0, w->cross_kv_b[i], 0, workspace, 4 * D, 0, 0, nullptr, 0, 0, 0, m * N, 4 * D, D, 1,
                CIR_ACT_NONE);
      if (rc == CIR_OK) rc = cir_kv_mxfp8_quantize(ctx, workspace, m * N, elems + (i * rn + r) * 4 * D, scales + (i * rn + r) * (4 * D / 32));
    }
  }
  ctx->gemm_force_pair = 0;
  return rc;
}

extern "C" size_t cir_stage2_kv_score_workspace_bytes(const cir_ctx* ctx, const cir_stage2_kv_cache* cache, int64_t T, int64_t C, int64_t Q,
                                                      int64_t L) {
  if (!cache) return 0;
  return s2_plan(ctx, nullptr, 0, T, C, Q, L, cache->num_tokens, kv_src(cache)).total;
}

extern "C" size_t cir_stage2_score_cached_workspace_bytes(const cir_ctx* ctx, int64_t T, int64_t Q, int64_t L, int64_t N) {
  return s2_plan(ctx, nullptr, 0, T, 0, Q, L, N, KV_CACHE).total;
}

extern "C" int cir_stage2_score_cached(cir_ctx* ctx, const cir_stage2_weights* w, const cir_stage2_kv_cache* cache,
                                       const int32_t* cand_list, int64_t C, const void* z_t, const int32_t* ids,
                                       const void* a0, const void* qc0,
                                       const int32_t* mask, int64_t Q, int64_t L,
                                       const int32_t* trip_query, const int32_t* trip_slot, int64_t T,
                                       const int32_t* attn_work, int64_t num_attn_work, const int32_t* attn_tiles, int64_t num_attn_tiles,
                                       const int32_t* attn_tiles_cls, int64_t num_attn_tiles_cls,
                                       float* scores, float* feats, void* workspace, size_t workspace_bytes) {
  CIR_ENTER(ctx);
  CIR_CHECK_ARG(cache != nullptr, "stage2_score_cached: cache is NULL");
  CIR_CHECK_ARG(kv_cache_serves(ctx, cache), "stage2_score_cached: cache format %d, context dtype %d", cache->dtype, ctx->dtype);
  CIR_CHECK_ARG(!a0 == !qc0, "stage2_score_cached: a0 and qc0 come as a pair");
  CIR_CHECK_ARG(T == 0 || a0 || (z_t && ids), "stage2_score_cached: z_t and ids are required without the a0 / qc0 prefix");
  CIR_CHECK_ARG(T == 0 || cache->rows >= 1, "stage2_score_cached: empty cache");
  return stage2_score_impl(ctx, w, nullptr, cand_list, C, a0 ? nullptr : z_t, a0 ? nullptr : ids, mask, Q, L, cache->num_tokens,
                           trip_query, trip_slot, T, attn_work, num_attn_work, attn_tiles, num_attn_tiles, attn_tiles_cls,
                           num_attn_tiles_cls, scores, feats, workspace, workspace_bytes, a0, qc0, cache);
}

// ------------------------------------------------------------------------------------------ re-ranking a device-resident top-K list
constexpr int64_t RERANK_MAX_T = 16384;          // one planning CTA (stage2_plan.cu)
constexpr int64_t RERANK_MAX_K = 2048;           // cir_rerank_sort

// slot / run_row / n_runs: MXFP8 caches only (cir_stage2_kv_runs), whose dequantised K/V of up to T runs sit in s2
struct RerankWs {
  int32_t *flat_pos, *kv_row, *trip_query, *tiles, *tiles_cls, *counts; float* sorted; void* s2; int32_t *slot, *run_row, *n_runs;
  size_t s2_bytes, total;
};
static RerankWs rerank_plan(const cir_ctx* ctx, void* ws, size_t bytes, int64_t Q, int64_t K, int64_t L, int64_t N, KvSrc src = KV_CACHE) {
  const int64_t T = Q * K;
  Bump b(ws, bytes);
  RerankWs w;
  w.flat_pos = (int32_t*)b.take(T * 4);
  w.kv_row = (int32_t*)b.take(T * 4);
  w.trip_query = (int32_t*)b.take(T * 4);
  w.tiles = (int32_t*)b.take(T * 16);
  w.tiles_cls = (int32_t*)b.take(T * 16);
  w.counts = (int32_t*)b.take(3 * 4);
  w.sorted = (float*)b.take(T * 4);
  w.s2_bytes = s2_plan(ctx, nullptr, 0, T, T, Q, L, N, src).total;
  w.s2 = b.take(w.s2_bytes);
  const bool runs = src == KV_CACHE_MXFP8;
  w.slot = runs ? (int32_t*)b.take(T * 4) : nullptr;
  w.run_row = runs ? (int32_t*)b.take(T * 4) : nullptr;
  w.n_runs = runs ? (int32_t*)b.take(4) : nullptr;
  w.total = align_up(b.off, 256);
  return w;
}
extern "C" size_t cir_stage2_rerank_cached_workspace_bytes(const cir_ctx* ctx, int64_t Q, int64_t K, int64_t L, int64_t N) {
  if (Q < 1 || K < 1 || L < 1 || N < 1) return 0;
  return rerank_plan(ctx, nullptr, 0, Q, K, L, N).total;
}
extern "C" size_t cir_stage2_kv_rerank_workspace_bytes(const cir_ctx* ctx, const cir_stage2_kv_cache* cache, int64_t Q, int64_t K, int64_t L) {
  if (!cache || Q < 1 || K < 1 || L < 1 || cache->num_tokens < 1) return 0;
  return rerank_plan(ctx, nullptr, 0, Q, K, L, cache->num_tokens, kv_src(cache)).total;
}

extern "C" int cir_stage2_rerank_cached(cir_ctx* ctx, const cir_stage2_weights* w, const cir_stage2_kv_cache* cache, const int32_t* cand,
                                        int64_t Q, int64_t K, const void* z_t, const int32_t* ids, const int32_t* mask, int64_t L,
                                        float* scores, int32_t* order, int32_t* ranked, int32_t* counts, void* workspace,
                                        size_t workspace_bytes) {
  CIR_ENTER(ctx);
  CIR_CHECK_ARG(w && cache && cand && z_t && ids && mask && scores && order, "stage2_rerank_cached: NULL argument");
  CIR_CHECK_ARG(kv_cache_serves(ctx, cache), "stage2_rerank_cached: cache format %d, context dtype %d", cache->dtype, ctx->dtype);
  CIR_CHECK_ARG(cache->rows >= 1, "stage2_rerank_cached: empty cache");
  CIR_CHECK_ARG(Q >= 1 && K >= 1 && K <= RERANK_MAX_K && Q * K <= RERANK_MAX_T,
                "stage2_rerank_cached: Q=%lld x K=%lld outside K <= %lld, Q*K <= %lld", (long long)Q, (long long)K,
                (long long)RERANK_MAX_K, (long long)RERANK_MAX_T);
  CIR_CHECK_ARG(L >= 1 && L <= 256, "stage2_rerank_cached: L=%lld outside [1, 256]", (long long)L);
  CIR_CHECK_ARG(cache->rows < (1ll << 18) - 1, "stage2_rerank_cached: a cache of %lld rows (at most 2^18 - 2)", (long long)cache->rows);
  const KvSrc src = kv_src(cache);
  const RerankWs ws = rerank_plan(ctx, workspace, workspace_bytes, Q, K, L, cache->num_tokens, src);
  if (workspace_bytes < ws.total) { cir_set_error("stage2_rerank_cached: workspace %zu < %zu", workspace_bytes, ws.total); return CIR_EWORKSPACE; }
  const int64_t T = Q * K;
  int32_t* cnt = counts ? counts : ws.counts;
  CIR_TRY(cir_stage2_plan_topk(ctx, cand, Q, K, L, cache->row0, cache->rows, ws.flat_pos, ws.kv_row, ws.trip_query, ws.tiles,
                               ws.tiles_cls, cnt));
  // one chunk of all T triplets, in the plan's candidate-major order: C is unused with a bf16 / fp32 cache and the tile lists are
  // bounded by T.  An MXFP8 cache needs the chunk's unique candidates: the runs of the sorted cache rows, at most T.
  const int32_t* trip_slot = ws.kv_row;
  if (src == KV_CACHE_MXFP8) {
    CIR_TRY(cir_stage2_kv_runs(ctx, ws.kv_row, cnt, T, cache->row0, ws.slot, ws.run_row, ws.n_runs));
    trip_slot = ws.slot;
  }
  CIR_TRY(stage2_score_impl(ctx, w, nullptr, ws.run_row, T, z_t, ids, mask, Q, L, cache->num_tokens, ws.trip_query, trip_slot, T,
                            nullptr, 0, ws.tiles, T, ws.tiles_cls, T, ws.sorted, nullptr, ws.s2, ws.s2_bytes, nullptr, nullptr, cache, cnt,
                            ws.n_runs));
  CIR_TRY(cir_stage2_scatter_scores(ctx, ws.sorted, ws.flat_pos, T, cnt, scores));
  CIR_TRY(cir_rerank_sort(ctx, scores, Q, K, order));
  if (ranked) CIR_TRY(cir_stage2_gather_ranked(ctx, cand, order, Q, K, ranked));
  return CIR_OK;
}
