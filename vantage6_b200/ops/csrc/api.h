// C ABI shared by the CUDA translation units and the pybind11 module (module.cpp).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#ifndef V6_MAX_PEERS
#define V6_MAX_PEERS 8
#endif

struct PeerTable { void* p[V6_MAX_PEERS]; };

// pad word layout (uint32 words inside each rank's signal pad, one 128 B line per group)
#define PAD_UPLOAD   0      // [0,8)   : rank p's weights for epoch e are final
#define PAD_BCAST    32     // [32,40) : reducer q has pushed its slice for epoch e
#define PAD_BARRIER  64     // [64,72) : generic barrier
#define PAD_SMALL    96     // [96,104): small_allreduce arrivals
#define PAD_ABORT    128    // host/any rank sets != 0 to abort all waits
#define PAD_STATUS   129    // kernel writes 1 here (own pad) when a wait timed out, 2 when a peer reducer reported a failed round
#define PAD_MISSING  130    // own pad: bitmask of ranks whose contribution never arrived (own waits OR'd with the peers' reports)
#define PAD_NI       136    // [136,144): n_i of rank p for this epoch (float bits), written by p into every reducer's pad
#define PAD_RFAIL    144    // [144,152): reducer q's round `epoch` failed (value = epoch), written by q into every pad
#define PAD_RMISS    152    // [152,160): the contributors reducer q missed (bitmask), written next to PAD_RFAIL

struct FedAvgParams {
    PeerTable upload;        // contribution buffer of every rank (peer VAs in my address space)
    PeerTable param_out;     // fp32 parameter buffer of every rank (push target)
    PeerTable shadow_out;    // optional bf16 shadow parameter buffer of every rank (or null)
    PeerTable pads;          // signal pad of every rank
    const void* upload_mc;   // multicast VA over all upload buffers (null -> P2P loads)
    void* param_mc;          // multicast VA over all param buffers (null -> P2P stores)
    void* shadow_mc;         // multicast VA over all shadow buffers (null -> P2P stores)
    float* w_global;         // fp32 master copy of my slice owner (full-size buffer, local)
    float* opt_m;            // server momentum / Adam m (local, full-size)
    float* opt_v;            // Adam v
    float weight[V6_MAX_PEERS];   // n_i of each rank (0 => not participating); ignored when dynamic_weights
    int dynamic_weights;     // 1: every rank only knows ITS n_i (my_weight); it travels to the reducers through PAD_NI
    float my_weight;
    long long lo, hi;        // my element slice [lo, hi) -- multiples of 8
    int rank, world;
    int n_reducers; uint32_t reducer_mask; uint32_t live_mask;   // reducer_mask bit p: rank p owns a slice;   // bit p: rank p is alive (waited for + pushed to); n_reducers:          // ranks [0, n_reducers) own a slice (1 = central server on GPU 0)
    uint32_t epoch;
    int upload_is_delta;     // 1: upload holds n_i*(w_i - w_g); 0: upload holds w_i (unscaled)
    int upload_prescaled;    // 1: contributions already multiplied by n_i (needed for multicast)
    int server_opt;          // 0 FedAvg (w += lr*d), 1 FedAvgM, 2 FedAdam
    float server_lr, beta1, beta2, eps, bias1, bias2;
    float inv_total;         // 1 / sum_i n_i over participants
    long long timeout_cycles;
    unsigned int* cta_counter;   // local scratch, zeroed by host once; self-resetting
    long long shadow_skip_lo, shadow_skip_hi;   // bf16 shadow elements [lo, hi) are NOT pushed to the peers (only written locally):
                                                // K1 delivers them, fused with the first GEMM that consumes them (gemm.cu)
};

struct SmallParams {
    PeerTable slots;      // payload slot of every rank (peer VAs), for this epoch's parity
    PeerTable pads;
    float weight[V6_MAX_PEERS];
    float* out;           // local result, n floats
    int n;                // floats, multiple of 4
    int rank, world;
    uint32_t epoch;
    float inv_total;
    long long timeout_cycles;
};

#define V6_MULTI_MAX 96
// multi-tensor gradient sink (optim.cu::multi_accum_kernel); passed by value as a kernel parameter (< 4 KB)
struct MultiAccumParams {
    const void* src[V6_MULTI_MAX];      // bf16 tensors, 16-byte aligned, dense
    long long dst_off[V6_MULTI_MAX];    // element offset into the fp32 destination (multiple of 8)
    long long numel[V6_MULTI_MAX];
    int count;
};

struct OptimParams {
    float* w;              // fp32 master weights (flat)
    const float* g;        // fp32 gradients (flat)
    float* m;              // momentum / Adam m
    float* v;              // Adam v (null for SGD)
    float* w_ref;          // (optional) global model received this round
    void* upload;          // (optional) contribution buffer (fp32 or bf16)
    void* shadow;           // (optional) bf16 copy of w
    const float* grad_scale_ptr;   // (optional) device scalar multiplied into g (loss-scale / clip)
    long long n;           // elements, multiple of 4
    float lr, momentum, dampening, weight_decay, beta1, beta2, eps, bias1, bias2;
    const float* bias_ptr;         // (optional) device [2]: Adam bias corrections computed on device (CUDA-graph safe)
    float contrib_scale;   // n_i
    const float* contrib_scale_ptr;   // (optional) device scalar that overrides contrib_scale (a captured graph reads the current n_i)
    int nesterov;
    int save_ref;          // 1: w_ref <- w(before step)
    int publish;           // 0 none, 1 delta fp32, 2 delta bf16, 3 weights fp32 (n_i * w_new)
    int first_momentum_step;   // torch semantics: buf = g on the very first step
};

#ifdef __cplusplus
extern "C" {
#endif
int v6_fedavg_round(const FedAvgParams* hp, int upload_dtype, int grid, cudaStream_t stream);
int v6_symm_barrier(const PeerTable* pads, int rank, int world, uint32_t epoch, long long timeout_cycles, cudaStream_t stream);
int v6_small_allreduce(const SmallParams* hp, cudaStream_t stream);
int v6_p2p_pull(const void* src_peer, void* dst_local, long long nbytes, cudaStream_t s);
int v6_mc_push(const void* src_local, void* mc_dst, long long nbytes, cudaStream_t s);
int v6_mc_reduce(const void* mc_src, void* dst_local, long long nbytes, cudaStream_t s);
int v6_flat_sgd(const OptimParams* hp, cudaStream_t s);
int v6_flat_adamw(const OptimParams* hp, cudaStream_t s);
int v6_delta_publish(const float* w, const float* ref, void* upload, long long n, float scale, int bf16_out, cudaStream_t s);
int v6_cast_bf16(const float* src, void* dst, long long n, cudaStream_t s);
int v6_adam_bias_update(int* step_counter, float beta1, float beta2, float* bias_out, cudaStream_t s);
int v6_clip_coef(const float* g, long long n, float max_norm, float* sumsq_scratch, float* coef, cudaStream_t s);
int v6_layernorm_fwd(const void* x, const void* residual, const float* gamma, const float* beta, void* y, void* res_out,
                     float* mean, float* rstd, int rows, int cols, float eps, int bf16, cudaStream_t s);
int v6_rmsnorm_fwd(const void* x, const void* residual, const float* gamma, void* y, void* res_out, float* rstd, int rows,
                   int cols, float eps, int bf16, cudaStream_t s);
int v6_layernorm_bwd(const void* dy, const void* x_in, const void* dres, const float* gamma, const float* mean,
                     const float* rstd, void* dx, float* dgamma, float* dbeta, float* scratch, int scratch_parts, int rows,
                     int cols, int accumulate, int bf16, cudaStream_t s);
int v6_rmsnorm_bwd(const void* dy, const void* x_in, const void* dres, const float* gamma, const float* rstd, void* dx,
                   float* dgamma, float* scratch, int scratch_parts, int rows, int cols, int accumulate, int bf16,
                   cudaStream_t s);
int v6_rope(void* q, void* k, const float* cos_t, const float* sin_t, const int* pos_ids, int B, int S, int Hq, int Hkv,
            int D, int inverse, cudaStream_t st);
int v6_glm_aggregate_update(const SmallParams* hp, const float* part, int nparts, int F, float rows, float lr, float* w,
                            float* loss_out, cudaStream_t stream);
int v6_glm_fold(const float* part, float* out, int nparts, int F, int rows, cudaStream_t s);
int v6_glm_logistic_grad_tc(const void* X, const float* y, const float* w, float* part, int max_parts, int rows, int F,
                            cudaStream_t s);
int v6_glm_logistic_grad(const void* X, const float* y, const float* w, float* part, int max_parts, float* out, int rows,
                         int F, int bf16, cudaStream_t s);
int v6_gemm_bf16(const void* A, const void* B, void* C, const float* bias, int M, int N, int K, int lda, int ldb, int ldc,
                 int act, cudaStream_t stream);
int v6_bcast_gemm_bf16(const void* A, void* B_local, const void* B_server_peer, void* C, const float* bias, int M, int N,
                       int K, int lda, int ldb, int ldc, int act, uint32_t* ready_flags, uint32_t epoch, cudaStream_t stream);
int v6_flash_attn_bwd(const void* q, const void* k, const void* v, const void* dout, const void* kt, const void* qt,
                      const void* dot, const float* lse2, const float* delta, void* dq, void* dk, void* dv, int B, int S,
                      int Hq, int Hkv, int D, float softmax_scale, int causal, cudaStream_t stream);
int v6_maxpool3x3s2_fwd(const void* x, void* y, void* idx, int N, int H, int W, int C, cudaStream_t s);
int v6_maxpool3x3s2_bwd(const void* dy, const void* idx, void* dx, int N, int H, int W, int C, cudaStream_t s);
int v6_image_normalize(const void* img, void* out, long long N, long long HW, float m0, float m1, float m2, float s0, float s1,
                       float s2, cudaStream_t s);
int v6_image_normalize_s2d(const void* img, void* out, int N, int H, int W, float m0, float m1, float m2, float s0, float s1,
                           float s2, cudaStream_t s);
int v6_stem_weight_s2d(const void* w, int w_is_bf16, void* ws, int O, cudaStream_t s);
int v6_stem_wgrad_d2s(const void* dws, float* dw, int O, int accumulate, cudaStream_t s);
int v6_bias_act_bwd(const void* dy, const void* pre, void* dpre, float* db, float* scratch, long long R, int C, int act_kind,
                    int accumulate, cudaStream_t s);
int v6_swiglu_fwd(const void* g, const void* u, void* h, long long n, cudaStream_t s);
int v6_swiglu_bwd(const void* dh, const void* g, const void* u, void* dg, void* du, long long n, cudaStream_t s);
long long v6_bn_scratch_floats();
int v6_multi_accum_bf16(const MultiAccumParams* p, float* dst, cudaStream_t s);
int v6_bn_fwd(const void* x, const void* res, const float* gamma, const float* beta, float* running_mean, float* running_var,
              long long* num_batches_tracked, void* y, void* relu_mask, float* mean, float* rstd, float* scale_bias,
              float* scratch, long long R, int C, float eps, float momentum, int relu, cudaStream_t s);
int v6_bn_apply(const void* x, const void* res, const float* scale, const float* bias, void* y, void* relu_mask, long long R, int C,
                int relu, cudaStream_t s);
int v6_ce_fwd(const void* logits, const long long* labels, float* lse, float* loss, int T, int V, long long ld, long long ignore_index,
              cudaStream_t s);
int v6_ce_bwd(void* logits, const long long* labels, const float* lse, const float* scale_ptr, int T, int V, int V_alloc, long long ld,
              long long ignore_index, cudaStream_t s);
int v6_bn_bwd(const void* dy, const void* relu_mask, const void* x, const float* gamma, const float* mean, const float* rstd, void* dx,
              void* dres, float* dgamma, float* dbeta, float* coef, float* scratch, long long R, int C, int relu,
              int accumulate, cudaStream_t s);
int v6_gemm2_bf16(const void* A, const void* B, void* C, const float* bias, int M, int N, int K, int lda, int ldb, int ldc,
                  int act, cudaStream_t stream);
int v6_gemm_smem_bytes();
int v6_bcast_push_gemm_bf16(const void* A, void* B_local, void* B_mc, void* C, const float* bias, int M, int N, int K, int lda, int ldb,
                            int ldc, int act, uint32_t* ready_flags, const PeerTable* flag_peers, int world, int is_owner,
                            uint32_t epoch, int own_nb_lo, int own_nb_hi, const uint32_t* epoch_ptr, uint32_t* status_ptr,
                            cudaStream_t stream);
int v6_flash_attn_fwd2_vmn(const void* q, const void* k, const void* v, void* o, float* lse, int B, int S, int Hq, int Hkv,
                           int D, long long ldq, long long ldk, long long ldv, float softmax_scale, int causal,
                           cudaStream_t stream);
int v6_flash_attn_fwd2(const void* q, const void* k, const void* vt, void* o, float* lse, int B, int S, int Hq, int Hkv,
                       int D, long long ldq, long long ldk, float softmax_scale, int causal, cudaStream_t stream);
int v6_flash_attn_fwd(const void* q, const void* k, const void* vt, void* o, float* lse, int B, int S, int Hq, int Hkv,
                      int D, long long ldq, long long ldk, float softmax_scale, int causal, cudaStream_t stream);
// symm.cpp
const char* v6_symm_last_error();
int v6_driver_available();
int v6_symm_init(int rank, int world, int device, const char* dir, int timeout_s);
int v6_symm_multicast_supported(int gid);
int v6_symm_alloc(int gid, size_t size, int want_multicast, uint64_t* peer_ptrs, uint64_t* mc_ptr, size_t* padded);
int v6_symm_barrier_host(int gid);
int v6_symm_free(int gid, int aid);
int v6_symm_finalize(int gid);
int v6_make_tmap_2d_bf16(void* out, uint64_t gptr, uint64_t rows, uint64_t cols, uint64_t row_stride_bytes,
                         uint32_t box_rows, uint32_t box_cols, int swizzle128);
int v6_make_tmap_tiled_bf16(void* out, uint64_t gptr, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                            const uint32_t* box, int swizzle128);
int v6_make_tmap_im2col_bf16(void* out, uint64_t gptr, uint64_t C, uint64_t W, uint64_t H, uint64_t N, int lower_w, int lower_h,
                             int upper_w, int upper_h, uint32_t channels, uint32_t pixels, uint32_t stride_w, uint32_t stride_h,
                             uint64_t pitch_w, uint64_t pitch_h, uint64_t pitch_n);
int v6_stem_wgrad_d2s_f32(const float* dws, float* dw, int O, int accumulate, cudaStream_t s);
// igemm.cu: implicit-GEMM convolution / linear-backward family
long long v6_igemm_scratch_floats();
int v6_conv_fprop(const void* x, const void* w, void* y, const float* bias, int act, int N, int H, int W, int Cin, int Cout, int R,
                  int S, int stride, int pad, const float* gamma, const float* beta, float* running_mean, float* running_var,
                  long long* num_batches_tracked, float* mean_out, float* rstd_out, float* scale_bias_out, float* scratch,
                  float eps, float momentum, int force_im2col, long long pitch_w, long long pitch_h, long long pitch_n,
                  cudaStream_t stream);
int v6_conv_dgrad(const void* dy, const void* w, void* dx, int N, int H, int W, int Cin, int Cout, int R, int S, int stride, int pad,
                  int force_im2col, const void* add_src, const void* add_mask, cudaStream_t stream);
int v6_conv_wgrad(const void* dy, const void* x, float* dw, int N, int H, int W, int Cin, int Cout, int R, int S, int stride, int pad,
                  float scale, int splits, int force_im2col, long long pitch_w, long long pitch_h, long long pitch_n,
                  float* ws, long long ws_floats, cudaStream_t stream);
long long v6_conv_wgrad_workspace(int N, int H, int W, int Cin, int Cout, int R, int S, int stride, int pad, int splits);
#ifdef __cplusplus
}
#endif
