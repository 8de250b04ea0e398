// Host launch API of the non-GEMM kernels (raw pointers + stream; the torch binding layer is bindings.cpp).
#pragma once
#include <cuda_runtime.h>

#include "seed.h"

namespace b200 {

// norm_embed.cu
void layer_norm_fwd(const void* x, const float* gamma, const float* beta, void* y, float* mean, float* rstd, int M,
                    int H, float eps, Seed seed, unsigned int stream, float p_drop, Fp8Out f8, cudaStream_t st);
int ln_bwd_workspace_floats(int M, int H);
void layer_norm_bwd(const void* dy, const void* x, const float* mean, const float* rstd, const float* gamma, void* dx,
                    void* dxd, float* dgamma, float* dbeta, float* dbias, float* workspace, int M, int H,
                    Seed seed, unsigned int drop_stream, unsigned int in_stream, float p_drop, Fp8Out f8,
                    cudaStream_t st, const uint8_t* keep_mask = nullptr);
void gelu_fwd(const void* x, void* y, long long n, Fp8Out f8, cudaStream_t st);
void dgelu_bwd(const void* dy, const void* x, void* dx, float* dbias, int M, int N, Fp8Out f8, cudaStream_t st);
// keep bits ([n_elems / 8] bytes, n_elems % 32 == 0) of the dropout stream (seed, stream): see dropout_mask_kernel
void dropout_mask(void* out, long long n_elems, Seed seed, unsigned int stream, float p_drop, cudaStream_t st);
void colsum_bf16(const void* x, int M, int N, int ld, float* out, cudaStream_t st);
void embedding_fwd(const int* ids, const int* seg, const void* word, const void* pos, const void* type,
                   const float* gamma, const float* beta, void* e_out, void* y, float* mean, float* rstd, int M, int S,
                   int H, float eps, Seed seed, unsigned int stream, float p_drop, cudaStream_t st);
void embedding_bwd_scatter(const void* de, const int* ids, const int* seg, float* gword, float* gpos, float* gtype,
                           int M, int S, int H, int type_rows, cudaStream_t st);
void mlm_compact(const int* labels, int B, int S, int max_pred, int* idx, int* tgt, int* count, cudaStream_t st);
void gather_rows(const void* src, const int* idx, void* dst, int n, int H, cudaStream_t st);
void scatter_rows(const void* src, const int* idx, void* dst, int n, int H, cudaStream_t st);

// loss.cu
void softmax_ce(void* logits, int ld, const int* targets, const int* count, float grad_scale, float* loss_out, int R,
                int V, cudaStream_t st);

// optim.cu   (dtype codes: 0 = fp32, 1 = bf16, 2 = fp16)
void mt_l2norm(int dtype, const long long* ptrs, const int* chunk_tensor, const long long* chunk_start,
               const int* chunk_len, int nchunks, float* per_tensor_sq, float* total_sq, cudaStream_t st);
void mt_scale(int in_dtype, int out_dtype, const long long* in_ptrs, const long long* out_ptrs,
              const int* chunk_tensor, const long long* chunk_start, const int* chunk_len, int nchunks,
              const float* scale_dev, float scale_host, int* overflow, cudaStream_t st);
void flat_sumsq(const float* g, long long n, const float* inv_scale, float* stats, float* found_inf, cudaStream_t st);
void flat_unscale(float* g, long long n, const float* inv_scale, float* found_inf, cudaStream_t st);
void arena_lamb(float* g, float* p, float* m, float* v, void* shadow, const int* chunk_tensor,
                const long long* chunk_start, const int* chunk_len, int nchunks, const int* decay_flag,
                int ntensors, float* stats, float* norms, const float* inv_scale, const float* found_inf,
                float lr, float beta1, float beta2, float eps, float weight_decay, int step, int bias_correction,
                int grad_averaging, float max_grad_norm, int adam_w_mode, int use_nvlamb, cudaStream_t st);
void arena_adam(float* g, float* p, float* m, float* v, void* shadow, const int* chunk_tensor,
                const long long* chunk_start, const int* chunk_len, int nchunks, const int* decay_flag,
                const float* inv_scale, const float* found_inf, float lr, float beta1, float beta2, float eps,
                float weight_decay, int step, int bias_correction, int adam_w_mode, cudaStream_t st);

// attention.cu
void attention_fwd(const void* qkv, const int* seqlens, void* ctx, float* lse, int B, int S, int h, int d,
                   float scale, Seed seed, unsigned int stream, float p_drop, Fp8Out f8, cudaStream_t st);
void attention_bwd(const void* qkv, const int* seqlens, const void* ctx, const void* dctx, const float* lse,
                   void* dqkv, float* delta_ws, float* dq_acc, int B, int S, int h, int d, float scale,
                   Seed seed, unsigned int stream, float p_drop, Fp8Out f8, cudaStream_t st);

// comm.cu -- fused peer-memory all-reduce + partitioned LAMB (one cooperative kernel per step)
struct FusedLambLaunch {
  int rank, world, use_multicast;
  const void* grad_ptrs[16]; const void* param_ptrs[16]; const void* shadow_ptrs[16];
  const void* pad_ptrs[16]; const void* flag_ptrs[16];
  void* grad_mc; void* param_mc; void* shadow_mc;
  float* m; float* v;
  long long numel, lo, hi;
  const int* chunk_tensor; const long long* chunk_start; const int* chunk_len; int nchunks, ntensors;
  const int* decay_flag;
  const int* prereduced = nullptr;   // per tensor flags: already reduced into the owner's arena by the wgrad GEMMs
  float* stats; float* norms; unsigned int* grid_bar;
  unsigned int epoch;
  float grad_mul, lr, beta1, beta2, eps, weight_decay, max_grad_norm;
  int step, bias_correction, grad_averaging, adam_w_mode, use_nvlamb;
  int push_master = 1;   // 0: peers receive only the bf16 shadow; the fp32 master stays with its owner
};
void fused_allreduce_lamb(const FusedLambLaunch& L, cudaStream_t st);

// in-place fp32 all-reduce (sum * scale) of a symmetric staging buffer, one kernel, P2P or NVLS multicast
struct PeerAllreduceLaunch {
  int rank, world, use_multicast;
  const void* buf_ptrs[16]; const void* flag_ptrs[16];
  void* buf_mc;
  unsigned int* grid_bar;
  unsigned int epoch;
  long long n;
  float scale;
};
void peer_allreduce(const PeerAllreduceLaunch& L, cudaStream_t st);

// loss.cu: NSP classifier + CE + backward in one launch
void nsp_head(const void* pooled_bf16, const void* w_bf16, const float* bias, const long long* labels, int B, int H,
              float grad_scale, float* loss_out, void* dz_bf16, float* dw, float* db, cudaStream_t st);

// gemm_mx.cu: block-scaled MXFP8 (e4m3 + one ue8m0 scale per 32 elements along K), NT layout
void mx_quantize(const void* x_bf16, void* q, void* sf, int R, int K, cudaStream_t st);
void gemm_mxfp8(const void* a, const void* sfa, const void* b, const void* sfb, void* out, int ldo, bool out_f32,
                const void* bias, int M, int N, int K, cudaStream_t st);

// fp8.cu: per-tensor scaled fp8 operand preparation; meta records are {amax, scale, inv_scale, _}
void fp8_quantize(const void* x_bf16, void* q, long long n, float* meta, bool e5m2, cudaStream_t st);
void fp8_amax(const void* x_bf16, long long n, float* meta, cudaStream_t st);
void fp8_update(float* meta, int nrec, const int* is_e5m2, float margin_pow2, cudaStream_t st);

}  // namespace b200
