// torch <-> kernel glue.  Every function takes torch tensors, checks what the kernels assume (device,
// dtype, contiguity, alignment) and launches on the current CUDA stream.
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/extension.h>

#include "gemm_sm100.h"
#include "kernels.h"

namespace {

using torch::Tensor;

inline cudaStream_t cur_stream() { return at::cuda::getCurrentCUDAStream().stream(); }
inline void check_bf16(const Tensor& t, const char* name) {
  TORCH_CHECK(t.is_cuda(), name, " must be a CUDA tensor");
  TORCH_CHECK(t.scalar_type() == at::kBFloat16, name, " must be bf16");
  TORCH_CHECK(t.stride(-1) == 1, name, " must have a unit inner stride");
  TORCH_CHECK(reinterpret_cast<uintptr_t>(t.data_ptr()) % 16 == 0, name, " must be 16-byte aligned");
}
// Device-resident dropout step counter mixed into every seed (set by the engine when it captures CUDA graphs:
// the pointer is baked into the captured launches, the counter is advanced inside the graph).
const unsigned long long* g_seed_step = nullptr;
Tensor g_seed_step_keepalive;
void set_seed_step(c10::optional<Tensor> t) {
  if (t.has_value() && t->defined()) {
    TORCH_CHECK(t->is_cuda() && t->scalar_type() == at::kLong && t->numel() == 1, "seed step must be a CUDA int64 scalar");
    g_seed_step_keepalive = *t;
    g_seed_step = reinterpret_cast<const unsigned long long*>(t->data_ptr<int64_t>());
  } else {
    g_seed_step = nullptr;
    g_seed_step_keepalive = Tensor();
  }
}
inline b200::Seed mk_seed(int64_t seed) { return b200::Seed{static_cast<unsigned long long>(seed), g_seed_step}; }

// Gradient arenas in NVLink symmetric memory: once registered, every fp32-accumulate GEMM whose output lies inside
// the local arena adds atomically (peers may be adding into it), and with `push` on the tile goes straight to
// the owner rank's arena (GEMM -> reduce-scatter in one kernel).
struct GradPeers {
  int world = 0, rank = 0, push = 0;
  int64_t numel = 0, per = 0;
  float* base[16] = {};
} g_grad_peers;
void set_grad_peers(int64_t world, int64_t rank, std::vector<int64_t> ptrs, int64_t numel, int64_t per) {
  TORCH_CHECK(world <= 16 && (int64_t)ptrs.size() == world, "set_grad_peers: <= 16 ranks, one pointer each");
  g_grad_peers = GradPeers();
  g_grad_peers.world = (int)world; g_grad_peers.rank = (int)rank; g_grad_peers.numel = numel; g_grad_peers.per = per;
  for (int i = 0; i < world; ++i) g_grad_peers.base[i] = reinterpret_cast<float*>(ptrs[i]);
}
void set_grad_push(bool on) { g_grad_peers.push = on ? 1 : 0; }

// optional fp8 side output: (q bytes, meta record, e5m2)
inline b200::Fp8Out mk_fp8(const c10::optional<Tensor>& q, const c10::optional<Tensor>& meta, bool e5m2, int64_t numel) {
  b200::Fp8Out f;
  if (q.has_value() && q->defined()) {
    TORCH_CHECK(meta.has_value() && meta->defined() && meta->scalar_type() == at::kFloat && meta->numel() >= 4, "fp8 meta");
    TORCH_CHECK(q->is_cuda() && q->is_contiguous() && q->element_size() == 1 && q->numel() == numel, "fp8 side output shape");
    f.q = reinterpret_cast<unsigned char*>(q->data_ptr());
    f.meta = meta->data_ptr<float>();
    f.e5m2 = e5m2 ? 1 : 0;
  }
  return f;
}

inline const void* opt_ptr(const c10::optional<Tensor>& t) { return t.has_value() && t->defined() ? t->data_ptr() : nullptr; }
inline float* opt_f32(const c10::optional<Tensor>& t) {
  if (!t.has_value() || !t->defined()) return nullptr;
  TORCH_CHECK(t->scalar_type() == at::kFloat && t->is_cuda(), "expected a CUDA fp32 tensor");
  return t->data_ptr<float>();
}

// D = epilogue(A op B).  a/b are 2-D bf16 (row stride arbitrary, multiple of 8 elements).
//   layout 0 (NT): a [M,K], b [N,K]     1 (NN): a [M,K], b [K,N]     2 (TN): a [K,M], b [K,N]
// fp8 mode (scale_a/scale_b given): a/b are 1-byte e4m3 (or e5m2, per flag) tensors, row strides multiples of 16,
// scale_* are the device inv_scale floats (views into the fp8 meta table); CTA-pair kernel only.
static inline bool p_drop_is_zero(double p) { return !(p > 0.0); }

void gemm(Tensor a, Tensor b, Tensor out, int64_t layout, int64_t epi, c10::optional<Tensor> bias,
          c10::optional<Tensor> res, c10::optional<Tensor> aux_out, int64_t k_splits, int64_t block_n, double alpha,
          double p_drop, int64_t seed, int64_t stream_id, c10::optional<Tensor> scale_a, c10::optional<Tensor> scale_b,
          bool a_e5m2, bool b_e5m2, bool allow_push, c10::optional<Tensor> colsum, c10::optional<Tensor> mask_out,
          c10::optional<Tensor> mask_in) {
  const bool fp8 = scale_a.has_value() && scale_a->defined();
  if (fp8) {
    TORCH_CHECK(a.is_cuda() && b.is_cuda() && a.element_size() == 1 && b.element_size() == 1 && a.stride(1) == 1 &&
                b.stride(1) == 1, "fp8 gemm operands must be CUDA 1-byte tensors with unit inner stride");
    TORCH_CHECK(scale_b.has_value() && scale_b->defined(), "fp8 gemm needs both dequantisation factors");
    TORCH_CHECK(a.stride(0) % 16 == 0 && b.stride(0) % 16 == 0 && reinterpret_cast<uintptr_t>(a.data_ptr()) % 16 == 0 &&
                reinterpret_cast<uintptr_t>(b.data_ptr()) % 16 == 0, "fp8 operands must be 16-byte aligned");
  } else {
    check_bf16(a, "a");
    check_bf16(b, "b");
  }
  TORCH_CHECK(a.dim() == 2 && b.dim() == 2 && out.dim() == 2, "gemm operands must be 2-D");
  c10::cuda::CUDAGuard guard(a.device());
  b200::GemmCall c;
  c.layout = (int)layout;
  c.epi = (int)epi;
  c.block_n = (int)block_n;
  int64_t M, N, K;
  if (layout == b200::GEMM_NT) { M = a.size(0); K = a.size(1); N = b.size(0); TORCH_CHECK(b.size(1) == K, "K mismatch"); }
  else if (layout == b200::GEMM_NN) { M = a.size(0); K = a.size(1); N = b.size(1); TORCH_CHECK(b.size(0) == K, "K mismatch"); }
  else { K = a.size(0); M = a.size(1); N = b.size(1); TORCH_CHECK(b.size(0) == K, "K mismatch"); }
  TORCH_CHECK(out.size(0) == M && out.size(1) == N, "output shape mismatch");
  TORCH_CHECK(a.stride(0) % 8 == 0 && b.stride(0) % 8 == 0, "row strides must be multiples of 8 elements");
  TORCH_CHECK(N % 8 == 0, "N must be a multiple of 8");
  const bool f32_out = (epi == b200::EPI_ACCUM_F32 || epi == b200::EPI_F32);
  TORCH_CHECK(out.is_cuda() && out.stride(1) == 1, "out must be CUDA with unit inner stride");
  TORCH_CHECK(out.scalar_type() == (f32_out ? at::kFloat : at::kBFloat16), "out dtype does not match the epilogue");
  TORCH_CHECK(reinterpret_cast<uintptr_t>(out.data_ptr()) % 16 == 0 && out.stride(0) % (f32_out ? 4 : 8) == 0,
              "out must be 16-byte aligned with an aligned row stride");
  c.M = (int)M; c.N = (int)N; c.K = (int)K;
  if (fp8) {
    c.fp8 = true; c.a_e5m2 = a_e5m2; c.b_e5m2 = b_e5m2;
    c.scale_a = opt_f32(scale_a); c.scale_b = opt_f32(scale_b);
  }
  c.A = a.data_ptr(); c.lda = (int)a.stride(0);
  c.B = b.data_ptr(); c.ldb = (int)b.stride(0);
  c.out = out.data_ptr(); c.ldo = (int)out.stride(0);
  if (aux_out.has_value() && aux_out->defined()) {
    check_bf16(*aux_out, "aux_out");
    TORCH_CHECK(aux_out->stride(0) == out.stride(0), "aux_out must share out's row stride");
    c.aux_out = aux_out->data_ptr();
  }
  if (bias.has_value() && bias->defined()) {
    check_bf16(*bias, "bias");
    TORCH_CHECK(bias->numel() == N, "bias length");
    c.bias = bias->data_ptr();
  }
  if (res.has_value() && res->defined()) {
    check_bf16(*res, "res");
    TORCH_CHECK(res->size(0) == M && res->size(1) == N && res->stride(0) % 8 == 0, "res shape");
    c.res = res->data_ptr(); c.ldr = (int)res->stride(0);
  }
  const bool needs_bias = epi == b200::EPI_BIAS || epi == b200::EPI_BIAS_GELU || epi == b200::EPI_BIAS_DROP_RES ||
                          epi == b200::EPI_BIAS_TANH || epi == b200::EPI_BIAS_GELU_DG;
  TORCH_CHECK(!needs_bias || c.bias != nullptr, "this epilogue needs a bias");
  TORCH_CHECK((epi != b200::EPI_BIAS_GELU && epi != b200::EPI_BIAS_GELU_DG) || c.aux_out != nullptr, "bias+gelu needs aux_out");
  TORCH_CHECK(epi != b200::EPI_DGELU || c.res != nullptr, "dgelu needs res (the pre-activation)");
  TORCH_CHECK(epi != b200::EPI_MUL || c.res != nullptr, "mul needs res");
  if (colsum.has_value() && colsum->defined()) {
    TORCH_CHECK(epi == b200::EPI_NONE || epi == b200::EPI_ADD || epi == b200::EPI_MUL,
                "column sums are fused into the plain / add / mul epilogues only");
    TORCH_CHECK(colsum->numel() == N && colsum->is_contiguous(), "colsum length");
    c.colsum = opt_f32(colsum);
  }
  TORCH_CHECK(epi != b200::EPI_BIAS_DROP_RES || c.res != nullptr, "bias+dropout+residual needs res");
  if (mask_out.has_value() && mask_out->defined()) {
    TORCH_CHECK(epi == b200::EPI_BIAS_DROP_RES && block_n == 512 && !p_drop_is_zero(p_drop), "mask_out: dropout epilogue of the CTA-pair kernel only");
    TORCH_CHECK(mask_out->is_cuda() && mask_out->scalar_type() == at::kByte && mask_out->is_contiguous() &&
                mask_out->numel() == M * (N / 8) && reinterpret_cast<uintptr_t>(mask_out->data_ptr()) % 16 == 0 && N % 128 == 0,
                "mask_out: uint8 [M, N / 8], 16-byte aligned, N % 128 == 0");
    c.mask_out = mask_out->data_ptr<uint8_t>();
  }
  if (mask_in.has_value() && mask_in->defined()) {
    TORCH_CHECK(epi == b200::EPI_BIAS_DROP_RES && block_n == 512 && !p_drop_is_zero(p_drop), "mask_in: dropout epilogue of the CTA-pair kernel only");
    TORCH_CHECK(mask_in->is_cuda() && mask_in->scalar_type() == at::kByte && mask_in->is_contiguous() &&
                mask_in->numel() == M * (N / 8) && reinterpret_cast<uintptr_t>(mask_in->data_ptr()) % 16 == 0 && N % 128 == 0,
                "mask_in: uint8 [M, N / 8], 16-byte aligned, N % 128 == 0");
    c.mask_in = mask_in->data_ptr<uint8_t>();
  }
  c.k_splits = (int)k_splits;
  c.alpha = (float)alpha;
  c.p_drop = (float)p_drop;
  c.seed = (unsigned long long)seed;
  c.seed_step = g_seed_step;
  if (epi == b200::EPI_ACCUM_F32 && g_grad_peers.world > 1) {
    const float* lo = g_grad_peers.base[g_grad_peers.rank];
    const float* o = reinterpret_cast<const float*>(out.data_ptr());
    if (o >= lo && o < lo + g_grad_peers.numel) {
      c.peer_world = g_grad_peers.world; c.peer_rank = g_grad_peers.rank;
      c.peer_push = (g_grad_peers.push && allow_push) ? 1 : 0;   // only tensors the fused step knows to be pre-reduced
      c.peer_off = (long long)(o - lo); c.peer_per = g_grad_peers.per;
      for (int i = 0; i < g_grad_peers.world; ++i) c.peer_base[i] = g_grad_peers.base[i];
    }
  }
  c.stream = (unsigned int)stream_id;
  b200::gemm_bf16(c, cur_stream());
}

void layer_norm_fwd(Tensor x, Tensor gamma, Tensor beta, Tensor y, c10::optional<Tensor> mean,
                    c10::optional<Tensor> rstd, double eps, double p_drop, int64_t seed, int64_t stream_id,
                    c10::optional<Tensor> q8, c10::optional<Tensor> meta8, bool e5m2) {
  check_bf16(x, "x"); check_bf16(y, "y");
  TORCH_CHECK(x.is_contiguous() && y.is_contiguous(), "x/y must be contiguous");
  const int H = (int)x.size(-1), M = (int)(x.numel() / H);
  TORCH_CHECK(H % 8 == 0, "hidden size must be a multiple of 8");
  c10::cuda::CUDAGuard guard(x.device());
  b200::layer_norm_fwd(x.data_ptr(), gamma.data_ptr<float>(), beta.data_ptr<float>(), y.data_ptr(), opt_f32(mean),
                       opt_f32(rstd), M, H, (float)eps, mk_seed(seed), (unsigned)stream_id, (float)p_drop,
                       mk_fp8(q8, meta8, e5m2, x.numel()), cur_stream());
}

int64_t ln_bwd_workspace(int64_t M, int64_t H) { return b200::ln_bwd_workspace_floats((int)M, (int)H); }

void layer_norm_bwd(Tensor dy, Tensor x, Tensor mean, Tensor rstd, Tensor gamma, Tensor dx, c10::optional<Tensor> dxd,
                    c10::optional<Tensor> dgamma, c10::optional<Tensor> dbeta, c10::optional<Tensor> dbias,
                    Tensor workspace, double p_drop, int64_t seed, int64_t drop_stream, int64_t in_stream,
                    c10::optional<Tensor> q8, c10::optional<Tensor> meta8, bool e5m2, c10::optional<Tensor> keep_mask) {
  check_bf16(dy, "dy"); check_bf16(x, "x"); check_bf16(dx, "dx");
  const int H = (int)x.size(-1), M = (int)(x.numel() / H);
  TORCH_CHECK(workspace.numel() >= b200::ln_bwd_workspace_floats(M, H), "LN workspace too small");
  c10::cuda::CUDAGuard guard(x.device());
  void* dxd_p = nullptr;
  if (dxd.has_value() && dxd->defined()) { check_bf16(*dxd, "dxd"); dxd_p = dxd->data_ptr(); }
  const uint8_t* km = nullptr;
  if (keep_mask.has_value() && keep_mask->defined()) {   // keep bits written by the producing GEMM (GemmCall::mask_out)
    TORCH_CHECK(keep_mask->is_cuda() && keep_mask->scalar_type() == at::kByte && keep_mask->is_contiguous() &&
                keep_mask->numel() == (int64_t)M * (H / 8), "keep_mask: uint8 [M, H / 8]");
    km = keep_mask->data_ptr<uint8_t>();
  }
  b200::layer_norm_bwd(dy.data_ptr(), x.data_ptr(), mean.data_ptr<float>(), rstd.data_ptr<float>(),
                       gamma.data_ptr<float>(), dx.data_ptr(), dxd_p, opt_f32(dgamma), opt_f32(dbeta), opt_f32(dbias),
                       workspace.data_ptr<float>(), M, H, mk_seed(seed), (unsigned)drop_stream,
                       (unsigned)in_stream, (float)p_drop, mk_fp8(q8, meta8, e5m2, x.numel()), cur_stream(), km);
}

void gelu_fwd(Tensor x, Tensor y, c10::optional<Tensor> q8, c10::optional<Tensor> meta8, bool e5m2) {
  check_bf16(x, "x"); check_bf16(y, "y");
  TORCH_CHECK(x.is_contiguous() && y.is_contiguous() && x.numel() == y.numel() && x.numel() % 8 == 0, "gelu_fwd shapes");
  c10::cuda::CUDAGuard guard(x.device());
  b200::gelu_fwd(x.data_ptr(), y.data_ptr(), x.numel(), mk_fp8(q8, meta8, e5m2, x.numel()), cur_stream());
}
void dgelu_bwd(Tensor dy, Tensor x, Tensor dx, c10::optional<Tensor> dbias, c10::optional<Tensor> q8,
               c10::optional<Tensor> meta8, bool e5m2) {
  check_bf16(dy, "dy"); check_bf16(x, "x"); check_bf16(dx, "dx");
  TORCH_CHECK(dy.dim() == 2 && dy.is_contiguous() && x.is_contiguous() && dx.is_contiguous() && dy.size(1) % 8 == 0,
              "dgelu_bwd: contiguous [M,N] with N % 8 == 0");
  c10::cuda::CUDAGuard guard(x.device());
  b200::dgelu_bwd(dy.data_ptr(), x.data_ptr(), dx.data_ptr(), opt_f32(dbias), (int)dy.size(0), (int)dy.size(1),
                  mk_fp8(q8, meta8, e5m2, dy.numel()), cur_stream());
}

void colsum(Tensor x, Tensor out) {
  check_bf16(x, "x");
  TORCH_CHECK(x.dim() == 2 && out.scalar_type() == at::kFloat && out.numel() == x.size(1), "colsum shapes");
  c10::cuda::CUDAGuard guard(x.device());
  b200::colsum_bf16(x.data_ptr(), (int)x.size(0), (int)x.size(1), (int)x.stride(0), out.data_ptr<float>(), cur_stream());
}

void embedding_fwd(Tensor ids, c10::optional<Tensor> seg, Tensor word, Tensor pos, c10::optional<Tensor> type,
                   Tensor gamma, Tensor beta, Tensor e_out, Tensor y, Tensor mean, Tensor rstd, int64_t S, double eps,
                   double p_drop, int64_t seed, int64_t stream_id) {
  TORCH_CHECK(ids.scalar_type() == at::kInt && ids.is_contiguous(), "ids must be contiguous int32");
  check_bf16(word, "word"); check_bf16(pos, "pos"); check_bf16(e_out, "e_out"); check_bf16(y, "y");
  const int H = (int)word.size(1), M = (int)ids.numel();
  c10::cuda::CUDAGuard guard(ids.device());
  const int* seg_p = nullptr;
  const void* type_p = nullptr;
  if (type.has_value() && type->defined()) {
    TORCH_CHECK(seg.has_value() && seg->scalar_type() == at::kInt, "segment ids must be int32");
    seg_p = seg->data_ptr<int>();
    type_p = type->data_ptr();
  }
  b200::embedding_fwd(ids.data_ptr<int>(), seg_p, word.data_ptr(), pos.data_ptr(), type_p, gamma.data_ptr<float>(),
                      beta.data_ptr<float>(), e_out.data_ptr(), y.data_ptr(), mean.data_ptr<float>(),
                      rstd.data_ptr<float>(), M, (int)S, H, (float)eps, mk_seed(seed), (unsigned)stream_id,
                      (float)p_drop, cur_stream());
}

void embedding_bwd_scatter(Tensor de, Tensor ids, c10::optional<Tensor> seg, Tensor gword, Tensor gpos,
                           c10::optional<Tensor> gtype, int64_t S) {
  check_bf16(de, "de");
  const int H = (int)de.size(-1), M = (int)ids.numel();
  c10::cuda::CUDAGuard guard(de.device());
  b200::embedding_bwd_scatter(de.data_ptr(), ids.data_ptr<int>(),
                              seg.has_value() && seg->defined() ? seg->data_ptr<int>() : nullptr,
                              gword.data_ptr<float>(), gpos.data_ptr<float>(), opt_f32(gtype), M, (int)S, H,
                              gtype.has_value() && gtype->defined() ? (int)gtype->size(0) : 0, cur_stream());
}

void mlm_compact(Tensor labels, int64_t max_pred, Tensor idx, Tensor tgt, Tensor count) {
  TORCH_CHECK(labels.scalar_type() == at::kInt && labels.dim() == 2 && labels.is_contiguous(), "labels: int32 [B,S]");
  c10::cuda::CUDAGuard guard(labels.device());
  b200::mlm_compact(labels.data_ptr<int>(), (int)labels.size(0), (int)labels.size(1), (int)max_pred,
                    idx.data_ptr<int>(), tgt.data_ptr<int>(), count.data_ptr<int>(), cur_stream());
}
void gather_rows(Tensor src, Tensor idx, Tensor dst) {
  check_bf16(src, "src"); check_bf16(dst, "dst");
  c10::cuda::CUDAGuard guard(src.device());
  b200::gather_rows(src.data_ptr(), idx.data_ptr<int>(), dst.data_ptr(), (int)idx.numel(), (int)src.size(-1), cur_stream());
}
void scatter_rows(Tensor src, Tensor idx, Tensor dst) {
  check_bf16(src, "src"); check_bf16(dst, "dst");
  c10::cuda::CUDAGuard guard(src.device());
  b200::scatter_rows(src.data_ptr(), idx.data_ptr<int>(), dst.data_ptr(), (int)idx.numel(), (int)src.size(-1), cur_stream());
}

void softmax_ce(Tensor logits, Tensor targets, Tensor count, double grad_scale, Tensor loss_out) {
  check_bf16(logits, "logits");
  TORCH_CHECK(logits.dim() == 2 && logits.size(1) % 8 == 0 && logits.stride(0) % 8 == 0, "logits: [R,V], V%8==0");
  c10::cuda::CUDAGuard guard(logits.device());
  b200::softmax_ce(logits.data_ptr(), (int)logits.stride(0), targets.data_ptr<int>(), count.data_ptr<int>(),
                   (float)grad_scale, loss_out.data_ptr<float>(), (int)logits.size(0), (int)logits.size(1), cur_stream());
}

inline int dtype_code(const Tensor& t) {
  if (t.scalar_type() == at::kFloat) return 0;
  if (t.scalar_type() == at::kBFloat16) return 1;
  if (t.scalar_type() == at::kHalf) return 2;
  TORCH_CHECK(false, "unsupported dtype for multi-tensor op");
  return -1;
}

void mt_l2norm(int64_t dtype, Tensor ptrs, Tensor chunk_tensor, Tensor chunk_start, Tensor chunk_len,
               c10::optional<Tensor> per_tensor_sq, Tensor total_sq) {
  c10::cuda::CUDAGuard guard(ptrs.device());
  b200::mt_l2norm((int)dtype, (const long long*)ptrs.data_ptr<int64_t>(), chunk_tensor.data_ptr<int>(),
                  (const long long*)chunk_start.data_ptr<int64_t>(), chunk_len.data_ptr<int>(),
                  (int)chunk_tensor.numel(), opt_f32(per_tensor_sq), total_sq.data_ptr<float>(), cur_stream());
}
void mt_scale(int64_t in_dtype, int64_t out_dtype, Tensor in_ptrs, Tensor out_ptrs, Tensor chunk_tensor,
              Tensor chunk_start, Tensor chunk_len, c10::optional<Tensor> scale_dev, double scale_host, Tensor overflow) {
  c10::cuda::CUDAGuard guard(in_ptrs.device());
  b200::mt_scale((int)in_dtype, (int)out_dtype, (const long long*)in_ptrs.data_ptr<int64_t>(),
                 (const long long*)out_ptrs.data_ptr<int64_t>(), chunk_tensor.data_ptr<int>(),
                 (const long long*)chunk_start.data_ptr<int64_t>(), chunk_len.data_ptr<int>(), (int)chunk_tensor.numel(),
                 opt_f32(scale_dev), (float)scale_host, overflow.data_ptr<int>(), cur_stream());
}
void flat_sumsq(Tensor g, c10::optional<Tensor> inv_scale, Tensor stats, c10::optional<Tensor> found_inf) {
  c10::cuda::CUDAGuard guard(g.device());
  TORCH_CHECK(g.numel() % 4 == 0, "arena size must be a multiple of 4");
  b200::flat_sumsq(g.data_ptr<float>(), g.numel(), opt_f32(inv_scale), stats.data_ptr<float>(), opt_f32(found_inf), cur_stream());
}
void flat_unscale(Tensor g, Tensor inv_scale, Tensor found_inf) {
  c10::cuda::CUDAGuard guard(g.device());
  b200::flat_unscale(g.data_ptr<float>(), g.numel(), inv_scale.data_ptr<float>(), found_inf.data_ptr<float>(), cur_stream());
}
void arena_lamb(Tensor g, Tensor p, Tensor m, Tensor v, c10::optional<Tensor> shadow, Tensor chunk_tensor,
                Tensor chunk_start, Tensor chunk_len, Tensor decay_flag, Tensor stats, Tensor norms,
                c10::optional<Tensor> inv_scale, c10::optional<Tensor> found_inf, double lr, double beta1, double beta2,
                double eps, double weight_decay, int64_t step, bool bias_correction, bool grad_averaging,
                double max_grad_norm, bool adam_w_mode, bool use_nvlamb) {
  c10::cuda::CUDAGuard guard(g.device());
  b200::arena_lamb(g.data_ptr<float>(), p.data_ptr<float>(), m.data_ptr<float>(), v.data_ptr<float>(),
                   shadow.has_value() && shadow->defined() ? shadow->data_ptr() : nullptr, chunk_tensor.data_ptr<int>(),
                   (const long long*)chunk_start.data_ptr<int64_t>(), chunk_len.data_ptr<int>(), (int)chunk_tensor.numel(),
                   decay_flag.data_ptr<int>(), (int)decay_flag.numel(), stats.data_ptr<float>(), norms.data_ptr<float>(),
                   opt_f32(inv_scale), opt_f32(found_inf), (float)lr, (float)beta1, (float)beta2, (float)eps,
                   (float)weight_decay, (int)step, bias_correction, grad_averaging, (float)max_grad_norm, adam_w_mode,
                   use_nvlamb, cur_stream());
}
void arena_adam(Tensor g, Tensor p, Tensor m, Tensor v, c10::optional<Tensor> shadow, Tensor chunk_tensor,
                Tensor chunk_start, Tensor chunk_len, Tensor decay_flag, c10::optional<Tensor> inv_scale,
                c10::optional<Tensor> found_inf, double lr, double beta1, double beta2, double eps, double weight_decay,
                int64_t step, bool bias_correction, bool adam_w_mode) {
  c10::cuda::CUDAGuard guard(g.device());
  b200::arena_adam(g.data_ptr<float>(), p.data_ptr<float>(), m.data_ptr<float>(), v.data_ptr<float>(),
                   shadow.has_value() && shadow->defined() ? shadow->data_ptr() : nullptr, chunk_tensor.data_ptr<int>(),
                   (const long long*)chunk_start.data_ptr<int64_t>(), chunk_len.data_ptr<int>(), (int)chunk_tensor.numel(),
                   decay_flag.data_ptr<int>(), opt_f32(inv_scale), opt_f32(found_inf), (float)lr, (float)beta1,
                   (float)beta2, (float)eps, (float)weight_decay, (int)step, bias_correction, adam_w_mode, cur_stream());
}

void attention_fwd(Tensor qkv, Tensor seqlens, Tensor ctx, Tensor lse, int64_t heads, double scale, double p_drop,
                   int64_t seed, int64_t stream_id, c10::optional<Tensor> q8, c10::optional<Tensor> meta8, bool e5m2) {
  check_bf16(qkv, "qkv"); check_bf16(ctx, "ctx");
  TORCH_CHECK(qkv.dim() == 3 && qkv.is_contiguous(), "qkv: contiguous [B,S,3H]");
  const int B = (int)qkv.size(0), S = (int)qkv.size(1), H = (int)qkv.size(2) / 3;
  c10::cuda::CUDAGuard guard(qkv.device());
  b200::attention_fwd(qkv.data_ptr(), seqlens.data_ptr<int>(), ctx.data_ptr(), lse.data_ptr<float>(), B, S, (int)heads,
                      H / (int)heads, (float)scale, mk_seed(seed), (unsigned)stream_id, (float)p_drop,
                      mk_fp8(q8, meta8, e5m2, ctx.numel()), cur_stream());
}
void attention_bwd(Tensor qkv, Tensor seqlens, Tensor ctx, Tensor dctx, Tensor lse, Tensor dqkv, Tensor delta_ws,
                   c10::optional<Tensor> dq_acc, int64_t heads, double scale, double p_drop, int64_t seed, int64_t stream_id,
                   c10::optional<Tensor> q8, c10::optional<Tensor> meta8, bool e5m2) {
  check_bf16(qkv, "qkv"); check_bf16(ctx, "ctx"); check_bf16(dctx, "dctx"); check_bf16(dqkv, "dqkv");
  TORCH_CHECK(qkv.is_contiguous() && ctx.is_contiguous() && dctx.is_contiguous() && dqkv.is_contiguous(), "attention_bwd needs contiguous tensors");
  const int B = (int)qkv.size(0), S = (int)qkv.size(1), H = (int)qkv.size(2) / 3;
  c10::cuda::CUDAGuard guard(qkv.device());
  b200::attention_bwd(qkv.data_ptr(), seqlens.data_ptr<int>(), ctx.data_ptr(), dctx.data_ptr(), lse.data_ptr<float>(),
                      dqkv.data_ptr(), delta_ws.data_ptr<float>(), opt_f32(dq_acc), B, S, (int)heads, H / (int)heads, (float)scale,
                      mk_seed(seed), (unsigned)stream_id, (float)p_drop, mk_fp8(q8, meta8, e5m2, dqkv.numel()), cur_stream());
}

void fused_allreduce_lamb(int64_t rank, int64_t world, bool use_multicast, std::vector<int64_t> grad_ptrs,
                          std::vector<int64_t> param_ptrs, std::vector<int64_t> shadow_ptrs, std::vector<int64_t> pad_ptrs,
                          std::vector<int64_t> flag_ptrs, int64_t grad_mc, int64_t param_mc, int64_t shadow_mc, Tensor m,
                          Tensor v, int64_t numel, int64_t lo, int64_t hi, Tensor chunk_tensor, Tensor chunk_start,
                          Tensor chunk_len, Tensor decay_flag, Tensor stats, Tensor norms, Tensor grid_bar, int64_t epoch,
                          double grad_mul, double lr, double beta1, double beta2, double eps, double weight_decay,
                          double max_grad_norm, int64_t step, bool bias_correction, bool grad_averaging,
                          bool adam_w_mode, bool use_nvlamb, bool push_master, c10::optional<Tensor> prereduced) {
  TORCH_CHECK((int64_t)grad_ptrs.size() == world && world <= 16, "peer pointer lists must have `world` (<= 16) entries");
  TORCH_CHECK(lo % 4 == 0 && hi % 4 == 0 && numel % 4 == 0, "shard bounds must be multiples of 4 elements");
  c10::cuda::CUDAGuard guard(m.device());
  b200::FusedLambLaunch L;
  L.rank = (int)rank; L.world = (int)world; L.use_multicast = use_multicast ? 1 : 0;
  for (int p = 0; p < world; ++p) {
    L.grad_ptrs[p] = reinterpret_cast<const void*>(grad_ptrs[p]);
    L.param_ptrs[p] = reinterpret_cast<const void*>(param_ptrs[p]);
    L.shadow_ptrs[p] = reinterpret_cast<const void*>(shadow_ptrs[p]);
    L.pad_ptrs[p] = reinterpret_cast<const void*>(pad_ptrs[p]);
    L.flag_ptrs[p] = reinterpret_cast<const void*>(flag_ptrs[p]);
  }
  L.grad_mc = reinterpret_cast<void*>(grad_mc); L.param_mc = reinterpret_cast<void*>(param_mc);
  L.shadow_mc = reinterpret_cast<void*>(shadow_mc);
  L.m = m.data_ptr<float>(); L.v = v.data_ptr<float>();
  L.numel = numel; L.lo = lo; L.hi = hi;
  L.chunk_tensor = chunk_tensor.data_ptr<int>(); L.chunk_start = (const long long*)chunk_start.data_ptr<int64_t>();
  L.chunk_len = chunk_len.data_ptr<int>(); L.nchunks = (int)chunk_tensor.numel(); L.ntensors = (int)decay_flag.numel();
  L.decay_flag = decay_flag.data_ptr<int>();
  TORCH_CHECK(stats.numel() >= 16, "fused_allreduce_lamb: stats needs 16 floats ([8..15] carry the in-kernel timeline)");
  L.stats = stats.data_ptr<float>(); L.norms = norms.data_ptr<float>();
  L.grid_bar = reinterpret_cast<unsigned int*>(grid_bar.data_ptr<int>());
  L.epoch = (unsigned int)epoch;
  L.grad_mul = (float)grad_mul; L.lr = (float)lr; L.beta1 = (float)beta1; L.beta2 = (float)beta2; L.eps = (float)eps;
  L.weight_decay = (float)weight_decay; L.max_grad_norm = (float)max_grad_norm; L.step = (int)step;
  L.bias_correction = bias_correction; L.grad_averaging = grad_averaging; L.adam_w_mode = adam_w_mode;
  L.use_nvlamb = use_nvlamb; L.push_master = push_master ? 1 : 0;
  if (prereduced.has_value() && prereduced->defined()) {
    TORCH_CHECK(prereduced->scalar_type() == at::kInt && prereduced->numel() == decay_flag.numel(), "prereduced flags");
    L.prereduced = prereduced->data_ptr<int>();
  }
  b200::fused_allreduce_lamb(L, cur_stream());
}

void nsp_head(Tensor pooled, Tensor w, Tensor bias, Tensor labels, double grad_scale, Tensor loss_out, Tensor dz, Tensor dw,
              Tensor db) {
  check_bf16(pooled, "pooled"); check_bf16(w, "w"); check_bf16(dz, "dz");
  TORCH_CHECK(pooled.dim() == 2 && pooled.is_contiguous() && dz.is_contiguous() && dz.sizes() == pooled.sizes(), "nsp_head: pooled/dz");
  const int64_t B = pooled.size(0), H = pooled.size(1);
  TORCH_CHECK(w.is_contiguous() && w.size(0) == 2 && w.size(1) == H, "nsp_head: w must be [2, H]");
  TORCH_CHECK(bias.scalar_type() == at::kFloat && bias.numel() == 2 && labels.scalar_type() == at::kLong && labels.numel() == B,
              "nsp_head: bias fp32 [2], labels int64 [B]");
  TORCH_CHECK(dw.scalar_type() == at::kFloat && dw.is_contiguous() && dw.numel() == 2 * H && db.scalar_type() == at::kFloat &&
              db.numel() == 2 && loss_out.scalar_type() == at::kFloat, "nsp_head: fp32 gradient / loss buffers");
  c10::cuda::CUDAGuard guard(pooled.device());
  b200::nsp_head(pooled.data_ptr(), w.data_ptr(), bias.data_ptr<float>(), reinterpret_cast<const long long*>(labels.data_ptr<int64_t>()), (int)B, (int)H,
                 (float)grad_scale, loss_out.data_ptr<float>(), dz.data_ptr(), dw.data_ptr<float>(), db.data_ptr<float>(),
                 cur_stream());
}

void peer_allreduce(int64_t rank, int64_t world, bool use_multicast, std::vector<int64_t> buf_ptrs,
                    std::vector<int64_t> flag_ptrs, int64_t buf_mc, Tensor grid_bar, int64_t epoch, int64_t n, double scale) {
  TORCH_CHECK((int64_t)buf_ptrs.size() == world && (int64_t)flag_ptrs.size() == world && world <= 16, "peer pointer lists");
  TORCH_CHECK(n % 4 == 0 && n > 0, "peer_allreduce: element count must be a positive multiple of 4");
  c10::cuda::CUDAGuard guard(grid_bar.device());
  b200::PeerAllreduceLaunch L;
  L.rank = (int)rank; L.world = (int)world; L.use_multicast = use_multicast ? 1 : 0;
  for (int p = 0; p < world; ++p) {
    L.buf_ptrs[p] = reinterpret_cast<const void*>(buf_ptrs[p]);
    L.flag_ptrs[p] = reinterpret_cast<const void*>(flag_ptrs[p]);
  }
  L.buf_mc = reinterpret_cast<void*>(buf_mc);
  L.grid_bar = reinterpret_cast<unsigned int*>(grid_bar.data_ptr<int>());
  L.epoch = (unsigned int)epoch; L.n = n; L.scale = (float)scale;
  b200::peer_allreduce(L, cur_stream());
}

// MXFP8: bf16 [R, K] -> e4m3 bytes [R, K] + ue8m0 block scales (one per 32 elements of K) in the tensor core's
// scale-factor layout [ceil(R/128)][K/128][512]
void mx_quantize(Tensor x, Tensor q, Tensor sf) {
  check_bf16(x, "x");
  TORCH_CHECK(x.dim() == 2 && x.is_contiguous() && x.size(1) % 128 == 0, "mx_quantize: contiguous [R, K] with K % 128 == 0");
  const int64_t R = x.size(0), K = x.size(1);
  TORCH_CHECK(q.is_cuda() && q.is_contiguous() && q.element_size() == 1 && q.numel() == R * K, "mx_quantize: q shape");
  TORCH_CHECK(sf.is_cuda() && sf.is_contiguous() && sf.element_size() == 1 &&
              sf.numel() == ((R + 127) / 128) * (K / 128) * 512, "mx_quantize: sf shape");
  c10::cuda::CUDAGuard guard(x.device());
  b200::mx_quantize(x.data_ptr(), q.data_ptr(), sf.data_ptr(), (int)R, (int)K, cur_stream());
}

// D[M,N] = A[M,K] . B[N,K]^T with block-scaled fp8 operands (tcgen05 kind::mxf8f6f4.block_scale)
void gemm_mxfp8(Tensor a, Tensor sfa, Tensor b, Tensor sfb, Tensor out, c10::optional<Tensor> bias) {
  TORCH_CHECK(a.dim() == 2 && b.dim() == 2 && a.is_contiguous() && b.is_contiguous() && a.element_size() == 1 &&
              b.element_size() == 1 && a.size(1) == b.size(1) && a.size(1) % 128 == 0, "gemm_mxfp8 operands");
  const int64_t M = a.size(0), N = b.size(0), K = a.size(1);
  TORCH_CHECK(sfa.numel() == ((M + 127) / 128) * (K / 128) * 512 && sfb.numel() == ((N + 127) / 128) * (K / 128) * 512,
              "gemm_mxfp8: scale-factor sizes");
  TORCH_CHECK(out.is_cuda() && out.dim() == 2 && out.size(0) == M && out.size(1) == N && out.stride(1) == 1 && N % 8 == 0,
              "gemm_mxfp8: out");
  const bool f32 = out.scalar_type() == at::kFloat;
  TORCH_CHECK(f32 || out.scalar_type() == at::kBFloat16, "gemm_mxfp8: out must be fp32 or bf16");
  const void* bp = nullptr;
  if (bias.has_value() && bias->defined()) { check_bf16(*bias, "bias"); TORCH_CHECK(bias->numel() == N, "bias"); bp = bias->data_ptr(); }
  c10::cuda::CUDAGuard guard(a.device());
  b200::gemm_mxfp8(a.data_ptr(), sfa.data_ptr(), b.data_ptr(), sfb.data_ptr(), out.data_ptr(), (int)out.stride(0), f32, bp,
                   (int)M, (int)N, (int)K, cur_stream());
}

void fp8_quantize(Tensor x, Tensor q, Tensor meta, bool e5m2) {
  check_bf16(x, "x");
  TORCH_CHECK(x.is_contiguous() && q.is_contiguous() && q.is_cuda() && q.element_size() == 1 && q.numel() == x.numel(),
              "fp8_quantize: q must be a contiguous 1-byte tensor of x's size");
  TORCH_CHECK(x.numel() % 16 == 0, "fp8_quantize: numel must be a multiple of 16");
  TORCH_CHECK(meta.scalar_type() == at::kFloat && meta.is_cuda() && meta.numel() >= 4, "fp8 meta record");
  c10::cuda::CUDAGuard guard(x.device());
  b200::fp8_quantize(x.data_ptr(), q.data_ptr(), x.numel(), meta.data_ptr<float>(), e5m2, cur_stream());
}

void fp8_amax(Tensor x, Tensor meta) {
  check_bf16(x, "x");
  TORCH_CHECK(x.is_contiguous() && x.numel() % 8 == 0, "fp8_amax: contiguous, numel % 8 == 0");
  c10::cuda::CUDAGuard guard(x.device());
  b200::fp8_amax(x.data_ptr(), x.numel(), meta.data_ptr<float>(), cur_stream());
}

void fp8_update(Tensor meta, Tensor is_e5m2, double margin_pow2) {
  TORCH_CHECK(meta.scalar_type() == at::kFloat && meta.is_cuda() && meta.is_contiguous() && meta.numel() % 4 == 0, "meta");
  TORCH_CHECK(is_e5m2.scalar_type() == at::kInt && is_e5m2.numel() * 4 == meta.numel(), "is_e5m2 flags");
  c10::cuda::CUDAGuard guard(meta.device());
  b200::fp8_update(meta.data_ptr<float>(), (int)(meta.numel() / 4), is_e5m2.data_ptr<int>(), (float)margin_pow2, cur_stream());
}

// measurement knobs of the pair GEMM (tools/gemm_lab.py): flags as in GemmArgs::lab, stats = int64 CUDA tensor [74 * 4] or None
void gemm_lab(int64_t flags, c10::optional<Tensor> stats) {
  unsigned long long* sp = nullptr;
  if (stats.has_value() && stats->defined()) {
    TORCH_CHECK(stats->is_cuda() && stats->scalar_type() == at::kLong && stats->numel() >= 74 * 12, "gemm_lab stats");
    sp = reinterpret_cast<unsigned long long*>(stats->data_ptr<int64_t>());
  }
  b200::gemm_lab((unsigned int)flags, sp);
}

// keep bits of the dropout stream (seed, stream) for a [.., N] tensor of `out.numel() * 8` elements (see dropout_mask_kernel)
void dropout_mask(Tensor out, double p_drop, int64_t seed, int64_t stream_id) {
  TORCH_CHECK(out.is_cuda() && out.scalar_type() == at::kByte && out.is_contiguous() && out.numel() % 4 == 0 &&
              reinterpret_cast<uintptr_t>(out.data_ptr()) % 16 == 0, "dropout_mask: uint8, contiguous, numel % 4 == 0");
  c10::cuda::CUDAGuard guard(out.device());
  b200::dropout_mask(out.data_ptr(), out.numel() * 8, mk_seed(seed), (unsigned)stream_id, (float)p_drop, cur_stream());
}

}  // namespace

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
  m.def("dropout_mask", &dropout_mask);
  m.def("gemm_lab", &gemm_lab);
  m.doc() = "bert_pytorch_b200 sm_100a kernels";
  m.def("gemm", &gemm);
  m.def("set_seed_step", &set_seed_step);
  m.def("set_grad_peers", &set_grad_peers);
  m.def("set_grad_push", &set_grad_push);
  m.def("peer_allreduce", &peer_allreduce);
  m.def("mx_quantize", &mx_quantize);
  m.def("gemm_mxfp8", &gemm_mxfp8);
  m.def("fp8_quantize", &fp8_quantize);
  m.def("fp8_amax", &fp8_amax);
  m.def("fp8_update", &fp8_update);
  m.def("layer_norm_fwd", &layer_norm_fwd);
  m.def("layer_norm_bwd", &layer_norm_bwd);
  m.def("ln_bwd_workspace", &ln_bwd_workspace);
  m.def("colsum", &colsum);
  m.def("gelu_fwd", &gelu_fwd);
  m.def("dgelu_bwd", &dgelu_bwd);
  m.def("embedding_fwd", &embedding_fwd);
  m.def("embedding_bwd_scatter", &embedding_bwd_scatter);
  m.def("mlm_compact", &mlm_compact);
  m.def("gather_rows", &gather_rows);
  m.def("scatter_rows", &scatter_rows);
  m.def("softmax_ce", &softmax_ce);
  m.def("nsp_head", &nsp_head);
  m.def("mt_l2norm", &mt_l2norm);
  m.def("mt_scale", &mt_scale);
  m.def("flat_sumsq", &flat_sumsq);
  m.def("flat_unscale", &flat_unscale);
  m.def("arena_lamb", &arena_lamb);
  m.def("arena_adam", &arena_adam);
  m.def("attention_fwd", &attention_fwd);
  m.def("attention_bwd", &attention_bwd);
  m.def("fused_allreduce_lamb", &fused_allreduce_lamb);
}
