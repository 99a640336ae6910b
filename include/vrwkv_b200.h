/*
 * vrwkv_b200.h — C ABI of the B200-native VisualRWKV hot path (libvrwkv_b200.so).
 *
 * Plain pointers and sizes only; no torch types.  All pointers are DEVICE pointers on the
 * current CUDA device unless stated otherwise.  `stream` is a cudaStream_t passed as void*
 * (NULL = legacy default stream, which is what the reference launches on,
 * VisualRWKV-v7/v7.00/cuda/wkv7_cuda.cu:133,137).
 *
 * Every entry point returns 0 on success or a negative VRWKV_E* code; the message of the last
 * failure on the calling thread is available from vrwkv_last_error().  Nothing here ever
 * falls back to a CPU path.
 *
 * "bf16" buffers are raw uint16_t storage of __nv_bfloat16.
 */
#ifndef VRWKV_B200_H
#define VRWKV_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VRWKV_OK 0
#define VRWKV_EINVAL (-1)  /* bad shape / alignment / null pointer */
#define VRWKV_ECUDA (-2)   /* CUDA runtime or driver error */
#define VRWKV_EUNSUP (-3)  /* shape outside what the kernels support (e.g. head size != 64) */

#define VRWKV_HEAD_SIZE 64 /* v7.00/src/model.py:69 hard-wires 64 */
#define VRWKV_CHUNK_LEN 16 /* v7.00/src/model.py:41 CHUNK_LEN */

const char* vrwkv_last_error(void);
int vrwkv_version(void);
/* Number of CUDA kernels this library has launched in this process (all entry points). */
unsigned long long vrwkv_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * WKV7 recurrence — replaces cuda_forward / cuda_backward
 * (VisualRWKV-v7/v7.00/cuda/wkv7_cuda.cu:132-138; bound by wkv7_op.cpp:7-19 as
 * torch.ops.wind_backstepping.{forward,backward}).
 *
 * w,q,k,v,a,b,y,dy,d*: bf16 [B,T,H,64] contiguous.  Argument order is the KERNEL order
 * (schema names w,q,k,v,z,a == kernel names w,q,k,v,a,b == python (w, r, k, v, -kk, kk*a)).
 * s : f32 [B,H,T/16,64,64]  state checkpoints, TRANSPOSED: s[b,h,c,j,i] = S_ij after step
 *     16c+15 (wkv7_cuda.cu:44-50).
 * sa: f32 [B,T,H,64]        sa[b,t,h,i] = sum_j a[t,j] S_ij (state BEFORE step t) (:27-32).
 * Requirements: T % 16 == 0 (model.py:49), all pointers 16-byte aligned, same device.
 * Caller allocates every output (model.py:52-54,63); the op keeps no state between calls.
 * ------------------------------------------------------------------------------------------ */
int vrwkv_wkv7_forward(int B, int T, int H, const uint16_t* w, const uint16_t* q,
                       const uint16_t* k, const uint16_t* v, const uint16_t* a,
                       const uint16_t* b, uint16_t* y, float* s, float* sa, void* stream);

int vrwkv_wkv7_backward(int B, int T, int H, const uint16_t* w, const uint16_t* q,
                        const uint16_t* k, const uint16_t* v, const uint16_t* a,
                        const uint16_t* b, const uint16_t* dy, const float* s, const float* sa,
                        uint16_t* dw, uint16_t* dq, uint16_t* dk, uint16_t* dv, uint16_t* da,
                        uint16_t* db, void* stream);

/* Stateful forward (SURVEY.md §8f-2; no reference counterpart for x070): as vrwkv_wkv7_forward
 * but the state starts from state_in (f32 [B,H,64,64], S_ij row-major; NULL = zeros) and the
 * final state is written to state_out (may alias state_in; NULL = not written).  s / sa may be
 * NULL (not written).  T may be any positive value when s == NULL. */
int vrwkv_wkv7_forward_state(int B, int T, int H, const uint16_t* w, const uint16_t* q,
                             const uint16_t* k, const uint16_t* v, const uint16_t* a,
                             const uint16_t* b, uint16_t* y, float* s, float* sa,
                             const float* state_in, float* state_out, void* stream);

/* Extended entry points: `flags` may carry VRWKV_WKV7_BOUNDED_DECAY, the caller's promise that exp(w) <= 0.607
 * everywhere — true for RWKV-7's w = -softplus(.) - 0.5 (VisualRWKV-v7/v7.00/src/model.py:176), i.e. for every call
 * RWKV_Tmix_x070 makes (model.py:190).  With it (and T % 64 == 0) the library evaluates the recurrence 64 steps at a
 * time on the tensor cores at fp32-level accuracy (every product is split into bf16 parts, csrc/wkv7_x6_common.cuh):
 * the outputs meet the same element-wise bounds as the step-by-step kernels.  Without it (the plain entry points above,
 * which is what torch.ops.wind_backstepping binds) the step-by-step kernels run for any w.  Same tensors, same contract. */
#define VRWKV_WKV7_BOUNDED_DECAY 1u
/* With BOUNDED_DECAY only (T % 64 == 0, no carried state): s is f32 [B,H,T/64,64,64] and holds one transposed state per
 * 64-step chunk (after step 64c+63) instead of the reference's T/16 checkpoints — all the chunked backward reads; a
 * quarter of the memory and of the forward's checkpoint writes.  Pass the same flag to forward_ex and backward_ex. */
#define VRWKV_WKV7_CHUNK_CHECKPOINTS 2u
/* With BOUNDED_DECAY: use the round-1 single-pass TF32 tensor-core kernels instead (faster products, but sa / s only
 * to ~5e-4 RMS: outside the north-star tolerance; kept for comparison, never a default). */
#define VRWKV_WKV7_TF32 4u
int vrwkv_wkv7_forward_ex(int B, int T, int H, const uint16_t* w, const uint16_t* q,
                          const uint16_t* k, const uint16_t* v, const uint16_t* a,
                          const uint16_t* b, uint16_t* y, float* s, float* sa,
                          const float* state_in, float* state_out, unsigned flags, void* stream);
int vrwkv_wkv7_backward_ex(int B, int T, int H, const uint16_t* w, const uint16_t* q,
                           const uint16_t* k, const uint16_t* v, const uint16_t* a,
                           const uint16_t* b, const uint16_t* dy, const float* s, const float* sa,
                           uint16_t* dw, uint16_t* dq, uint16_t* dk, uint16_t* dv, uint16_t* da,
                           uint16_t* db, unsigned flags, void* stream);
/* Chunk cache: with flags = BOUNDED_DECAY | CHUNK_CHECKPOINTS (T % 64 == 0, no carried state, s and sa required),
 * forward_cache is forward_ex that also writes `cache`, and backward_cache is backward_ex that reads it back instead of
 * recomputing what the forward already had: the masked 64x64 chunk matrices and the triangular inverse of each chunk.
 * The cache holds vrwkv_wkv7_cache_bytes(B, T, H) bytes (64 KB per 64-step chunk of each (batch, head); 0 when
 * T % 64 != 0), 128-byte aligned, and is only meaningful to backward_cache on the same inputs, s and sa. */
size_t vrwkv_wkv7_cache_bytes(int B, int T, int H);
int vrwkv_wkv7_forward_cache(int B, int T, int H, const uint16_t* w, const uint16_t* q,
                             const uint16_t* k, const uint16_t* v, const uint16_t* a,
                             const uint16_t* b, uint16_t* y, float* s, float* sa, void* cache,
                             unsigned flags, void* stream);
int vrwkv_wkv7_backward_cache(int B, int T, int H, const uint16_t* w, const uint16_t* q,
                              const uint16_t* k, const uint16_t* v, const uint16_t* a,
                              const uint16_t* b, const uint16_t* dy, const float* s, const float* sa,
                              const void* cache, uint16_t* dw, uint16_t* dq, uint16_t* dk, uint16_t* dv,
                              uint16_t* da, uint16_t* db, unsigned flags, void* stream);
/* Synchronises the device and fails (VRWKV_EINVAL) if a chunked kernel saw decay outside the promised range since
 * the last check; the flag is cleared. */
int vrwkv_wkv7_domain_check(void);
/* Development aid: per-phase clock stamps of the chunked forward kernel are written to buf (NULL disables). */
int vrwkv_wkv7_chunk_debug(float* buf);

/* Kernel-variant selection for benchmarking (0 = default heuristic; forward 1/2 step-by-step, 3 TF32 chunked, 6 x6
 * chunk-parallel; backward 1/2 step-by-step, 3/4 TF32 dS scan + step-by-step kernel on 64-step segments, 5 TF32 dS scan
 * + chunked tensor-core kernel, 7 x3 chunked). Thread-safe, process-wide. */
int vrwkv_wkv7_set_variant(int fwd_variant, int bwd_variant);


/* ------------------------------------------------------------------------------------------
 * Fused row-wise kernels of the RWKV-7 block (all tensors bf16 row-major [rows, C], rows = B*T,
 * C a multiple of 64 and <= 2048; per-channel parameters bf16 [C]).  Parameter gradients leave as
 * fp32 per-CTA partial rows `partial[blocks][n][C]` that the caller sums over `blocks`
 * (blocks = vrwkv_ln_mix_blocks(rows) / vrwkv_tmix_blocks(rows)).
 * ------------------------------------------------------------------------------------------ */

/* LayerNorm (+ token shift + NMIX lerps) — replaces ln1/ln2 + nn.ZeroPad2d((0,0,1,-1)) + the six / one
 * `x + xx * x_*` mixes (v7.00/src/model.py:149,166-173,222-224,250,252) and the plain LayerNorms (:248,323,338).
 * nmix in {0,1,6}; gamma == beta == NULL: input already normalised (mix only); out[m] = h + (shift(h) - h) coef[m].
 * coef / out / dout are HOST arrays of nmix device pointers.  stats: f32 [rows,2] (mean, rstd). */
int vrwkv_ln_mix_blocks(int rows);
int vrwkv_ln_mix_blocks2(int rows, int C);   /* partial rows vrwkv_ln_mix_backward writes for this shape (use this one) */
int vrwkv_ln_mix_forward(int rows, int T, int C, int nmix, float eps, const uint16_t* x, const uint16_t* gamma,
                         const uint16_t* beta, const uint16_t* const* coef, uint16_t* const* out, uint16_t* h_out,
                         float* stats, void* stream);
/* dx = LN-backward(sum over mixes) [+ dresid]; partial rows: dgamma, dbeta, dcoef[0..nmix). dh: gradient of the LN
 * output when nmix == 0. */
int vrwkv_ln_mix_backward(int rows, int T, int C, int nmix, const uint16_t* x, const float* stats, const uint16_t* gamma,
                          const uint16_t* beta, const uint16_t* const* coef, const uint16_t* const* dout,
                          const uint16_t* dh, const uint16_t* dresid, uint16_t* dx, float* partial, void* stream);

/* tmix_mid — model.py:176-190: w = -softplus(-(w0+ww)) - 0.5 ; a = sigmoid(a0+aa) ; v2 = v + (vfirst - v) sigmoid(v0+vv)
 * (vfirst == NULL for layer 0: v2 = v) ; kk = normalize_head(k*k_k) ; k2 = k (1 + (a-1) k_a) ; nkk = -kk ; kka = kk*a. */
int vrwkv_tmix_blocks(int rows);
int vrwkv_tmix_mid_forward(int rows, int C, const uint16_t* k, const uint16_t* v, const uint16_t* vfirst, const uint16_t* ww,
                           const uint16_t* aa, const uint16_t* vv, const uint16_t* w0, const uint16_t* a0, const uint16_t* v0,
                           const uint16_t* k_k, const uint16_t* k_a, uint16_t* w, uint16_t* k2, uint16_t* v2, uint16_t* nkk,
                           uint16_t* kka, void* stream);
/* partial rows: dw0, da0, dv0, dk_k, dk_a.  dk2b / dv2b: optional second gradient contributions (added to dk2 / dv2). */
int vrwkv_tmix_mid_backward(int rows, int C, const uint16_t* k, const uint16_t* v, const uint16_t* vfirst, const uint16_t* ww,
                            const uint16_t* aa, const uint16_t* vv, const uint16_t* w0, const uint16_t* a0, const uint16_t* v0,
                            const uint16_t* k_k, const uint16_t* k_a, const uint16_t* dw, const uint16_t* dk2,
                            const uint16_t* dv2, const uint16_t* dnkk, const uint16_t* dkka, const uint16_t* dk2b,
                            const uint16_t* dv2b, uint16_t* dk, uint16_t* dv, uint16_t* dvfirst, uint16_t* dww, uint16_t* daa,
                            uint16_t* dvv, float* partial, void* stream);

/* tmix_post — model.py:191-194: z = (GroupNorm_H(y; eps) + (sum_head r k2 r_k) v2) * g   (the input of `output`). */
int vrwkv_tmix_post_forward(int rows, int C, float eps, const uint16_t* y, const uint16_t* r, const uint16_t* k2,
                            const uint16_t* v2, const uint16_t* g, const uint16_t* gamma, const uint16_t* beta,
                            const uint16_t* r_k, uint16_t* z, void* stream);
/* partial rows: dgamma, dbeta, dr_k */
int vrwkv_tmix_post_backward(int rows, int C, float eps, const uint16_t* y, const uint16_t* r, const uint16_t* k2,
                             const uint16_t* v2, const uint16_t* g, const uint16_t* gamma, const uint16_t* beta,
                             const uint16_t* r_k, const uint16_t* dz, uint16_t* dy, uint16_t* dr, uint16_t* dk2, uint16_t* dv2,
                             uint16_t* dg, float* partial, void* stream);

/* out[n*C] (bf16) = sum_b partial[b][n*C]: second stage of the parameter gradients of the kernels above. */
int vrwkv_reduce_partials(int nblocks, int n_times_c, const float* partial, uint16_t* out, void* stream);

/* relu(x)^2 — model.py:225 (n elements, n % 8 == 0). The *_from_act backward needs only y = relu(x)^2. */
int vrwkv_relu_sq_forward(size_t n, const uint16_t* x, uint16_t* y, void* stream);
int vrwkv_relu_sq_backward(size_t n, const uint16_t* x, const uint16_t* dy, uint16_t* dx, void* stream);
int vrwkv_relu_sq_backward_from_act(size_t n, const uint16_t* y, const uint16_t* dy, uint16_t* dx, void* stream);

/* Shifted cross-entropy + L2Wrap over logits [rows = B*T, V] (bf16) — model.py:418-434, 257-271.
 * forward: lse/rowmax/nll f32 [rows], argmax i32 [rows]; the target of row (b,t) is labels[b,t+1] (int64 [B,T]).
 * backward: overwrites `logits_inout` with wrow[row] * (softmax - onehot(target)) + l2 * rowmax * onehot(argmax). */
int vrwkv_ce_forward(int rows, int T, int V, int ignore_index, const uint16_t* logits, const long long* labels, float* lse,
                     float* rowmax, int* argmax, float* nll, void* stream);
int vrwkv_ce_backward(int rows, int T, int V, int ignore_index, uint16_t* logits_inout, const long long* labels,
                      const float* lse, const float* rowmax, const int* argmax, const float* wrow, float l2, void* stream);

/* bf16 GEMM on the tcgen05 tensor cores: C[M,N] = epilogue(A[M,K] . B[N,K]^T), fp32 accumulate in TMEM.
 * epilogue 0: none (receptance/key/value, model.py:175-178); 1: relu(.)^2 (channel-mix key, :225);
 * 2: + R[M,N] (output / value projections with the residual add, :194,227,251-252).  K % 64 == 0, N % 128 == 0. */
int vrwkv_gemm_bf16_tn(int M, int N, int K, const uint16_t* A, const uint16_t* B, uint16_t* C, int epilogue,
                       const uint16_t* R, void* stream);

/* CTA-pair GEMM (tcgen05.mma.cta_group::2, 256-row tiles across two SMs), every layout of the forward and backward
 * products of model.py:175-194,225-227,325:   C[g] = epilogue(op(A[g]) . op(B[g])), g < ngroups problems of one shape in
 * one launch.  layout bit 0: A is [K,M] (else [M,K]); bit 1: B is [K,N] (else [N,K], the nn.Linear weight layout).
 * epilogue 0 none, 1 relu(.)^2, 2 + R[g], 4 (.) * 2 sqrt(R[g]) (backward of relu^2 from the saved activation),
 * 5 + bias[g][n], 6 tanh-GELU(. + bias), 7 . + bias + R[g][row % r_rows] (the SigLIP tower's Linear layers),
 * 8 act[g](.) with act 0 none / 1 tanh / 2 sigmoid, 9 (.) * act[g]'(R[g]) from the saved output (the LoRA branches).
 * ksplit > 1 slices the contraction (weight gradients over the 16384 token rows): slices meet in an internal fp32
 * workspace and the last one writes the bf16 result; c_transposed[g] != 0 stores C[g] as [N,M] (plain epilogue only).
 * K % (64 ksplit) == 0, N % 128 == 0, M % 8 == 0 for layout bit 0.
 * dims (optional, 3 ints per group: Mg, Ng, Kg <= M, N, K, multiples of 8): the group's tensors are exactly that
 * large (row strides Mg/Ng/Kg); the launch tiles (M, N, K) and the loads zero-fill / the stores clip beyond them, so
 * LoRA branches of different rank share a launch unpadded. */
int vrwkv_gemm2_bf16_grouped(int M, int N, int K, int ngroups, const uint16_t* const* A, const uint16_t* const* B,
                             uint16_t* const* C, const uint16_t* const* R, const int* c_transposed, int layout,
                             int epilogue, int ksplit, const uint16_t* const* bias, int r_rows, const int* act, const int* dims, void* stream);
int vrwkv_gemm2_bf16(int M, int N, int K, const uint16_t* A, const uint16_t* B, uint16_t* C, int layout, int epilogue,
                     const uint16_t* R, int ksplit, void* stream);

/* VisualRWKV.preparing_embedding (model.py:473-494): out[t] = emb[ids[t]], except that the k-th token (row-major over the
 * batch) with ids == image_token_index takes feats[k] (bit-exact row copies).  *n_slots_out (device int, may be NULL)
 * receives the number of image-token slots; slots beyond nfeat keep the embedding row.  The backward gathers dout rows
 * back into feature order (rows without a slot are zero).  D % 8 == 0. */
int vrwkv_embed_scatter_forward(int ntok, int D, int nfeat, long long image_token_index, const long long* ids,
                                const uint16_t* emb, const uint16_t* feats, uint16_t* out, int* n_slots_out, void* stream);
int vrwkv_embed_scatter_backward(int ntok, int D, int nfeat, long long image_token_index, const long long* ids,
                                 const uint16_t* dout, uint16_t* dfeats, void* stream);
/* VisualRWKV.adaptive_pooling (model.py:442-447): x [N, hw*hw, D] -> AdaptiveAvgPool2d(out) -> y [N, out*out, D]. */
int vrwkv_adaptive_pool(int N, int hw, int out, int D, const uint16_t* x, uint16_t* y, void* stream);

/* SigLIP self-attention, forward only (transformers SiglipAttention as called by VisualRWKV-v7/v7.01/src/model.py:347-352,
 * 448-454): q, k, v, o are [N*S, 64*H] bf16 (heads side by side); softmax(q k^T / 8) v per (image, head).  S <= 256. */
int vrwkv_vit_attention(int N, int S, int H, const uint16_t* q, const uint16_t* k, const uint16_t* v, uint16_t* o, void* stream);
/* pixels [N,3,Hp*P,Wp*P] -> patch rows [N*Hp*Wp, 3*P*P] in Conv2d weight order (the patch embedding becomes a GEMM). */
int vrwkv_im2col_patches(int N, int Hp, int Wp, int P, const uint16_t* pixels, uint16_t* out, void* stream);
/* MLPWithContextGating's gate (model.py:335-338): h = x * sigmoid(g), and its backward (dx may be NULL). n % 8 == 0. */
int vrwkv_sigmul_forward(size_t n, const uint16_t* x, const uint16_t* g, uint16_t* h, void* stream);
int vrwkv_sigmul_backward(size_t n, const uint16_t* x, const uint16_t* g, const uint16_t* dh, uint16_t* dx, uint16_t* dg, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Optimizer step of the training loop: AdamW over bf16 parameters with fp32 master weights and moments (the reference
 * configures DeepSpeed FusedAdam in adam_w_mode over bf16 weights, v7.00/src/model.py:376-410).  One multi-tensor pass:
 * reads the bf16 gradient and the fp32 state, writes the state and the bf16 parameter (28 bytes per parameter).
 * tensors: device array of 32-byte records {bf16* param, const bf16* grad, int64 state_off, int64 numel};
 * chunks: device array of int2 {tensor index, chunk index}, chunk = vrwkv_adamw_chunk() elements;
 * step: device int, incremented before the update (bias correction), so a call is CUDA-graph capturable;
 * lr_dev: optional device float overriding lr;  grad_scale multiplies the gradient (e.g. 1 / world size).
 * --------------------------------------------------------------------------------------------- */
int vrwkv_adamw_chunk(void);
int vrwkv_adamw_step(int nchunks, const void* tensors, const void* chunks, float* master, float* exp_avg, float* exp_avg_sq,
                     int* step, const float* lr_dev, float lr, float beta1, float beta2, float eps, float weight_decay,
                     float grad_scale, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VRWKV_B200_H */
