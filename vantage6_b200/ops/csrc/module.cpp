// pybind11 bindings (CPython C-API, no torch headers): every function takes raw device
// pointers (tensor.data_ptr()) and a CUDA stream handle (torch.cuda.current_stream().cuda_stream).
// Python-side wrappers with shape/dtype checks and autograd live in vantage6_b200/ops/*.py.
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include <algorithm>
#include <stdexcept>
#include <string>
#include <vector>

#include "api.h"

namespace py = pybind11;
using u64 = uint64_t;

static void check(int rc, const char* what) {
    if (rc == 0) return;
    std::string msg = std::string(what) + " failed: ";
    if (rc > 0) msg += cudaGetErrorString((cudaError_t)rc);
    else msg += v6_symm_last_error();
    throw std::runtime_error(msg);
}
static inline cudaStream_t S(u64 s) { return reinterpret_cast<cudaStream_t>(s); }
template <typename T> static inline T* P(u64 p) { return reinterpret_cast<T*>(p); }
static PeerTable table(const std::vector<u64>& v) {
    PeerTable t;
    for (int i = 0; i < V6_MAX_PEERS; ++i) t.p[i] = i < (int)v.size() ? reinterpret_cast<void*>(v[i]) : nullptr;
    return t;
}

PYBIND11_MODULE(_C, m) {
    m.doc() = "vantage6_b200 native sm_100a kernels + NVLink symmetric heap";
    m.attr("MAX_PEERS") = V6_MAX_PEERS;
    m.attr("PAD_WORDS") = 256;
    m.attr("PAD_ABORT") = PAD_ABORT;
    m.attr("PAD_STATUS") = PAD_STATUS;
    m.attr("PAD_MISSING") = PAD_MISSING;

    // ------------------------------------------------------------------ symmetric heap
    m.def("driver_available", [] { return v6_driver_available() != 0; });
    m.def("symm_init", [](int rank, int world, int device, const std::string& dir, int timeout_s) {
        int gid;
        { py::gil_scoped_release nogil; gid = v6_symm_init(rank, world, device, dir.c_str(), timeout_s); }
        if (gid < 0) throw std::runtime_error(std::string("symm_init: ") + v6_symm_last_error());
        return gid;
    });
    m.def("symm_multicast_supported", &v6_symm_multicast_supported);
    m.def("symm_alloc", [](int gid, size_t size, bool want_mc) {
        uint64_t ptrs[V6_MAX_PEERS] = {0};
        uint64_t mc = 0;
        size_t padded = 0;
        int aid;
        { py::gil_scoped_release nogil; aid = v6_symm_alloc(gid, size, want_mc ? 1 : 0, ptrs, &mc, &padded); }
        if (aid < 0) throw std::runtime_error(std::string("symm_alloc: ") + v6_symm_last_error());
        std::vector<u64> v(ptrs, ptrs + V6_MAX_PEERS);
        return py::make_tuple(aid, v, mc, padded);
    });
    m.def("symm_barrier_host", [](int gid) { py::gil_scoped_release nogil; check(v6_symm_barrier_host(gid), "symm_barrier_host"); });
    m.def("symm_free", [](int gid, int aid) { py::gil_scoped_release nogil; v6_symm_free(gid, aid); });
    m.def("symm_finalize", [](int gid) { py::gil_scoped_release nogil; v6_symm_finalize(gid); });

    // ------------------------------------------------------------------ K2 / K3 / barrier
    m.def("fedavg_round",
          [](const std::vector<u64>& upload, const std::vector<u64>& param_out, const std::vector<u64>& shadow_out,
             const std::vector<u64>& pads, u64 upload_mc, u64 param_mc, u64 shadow_mc, u64 w_global, u64 opt_m, u64 opt_v,
             const std::vector<float>& weight, long long lo, long long hi, int rank, int world, int n_reducers,
             uint32_t live_mask, uint32_t epoch, bool upload_is_delta, bool upload_prescaled, int server_opt, float server_lr, float beta1,
             float beta2, float eps, float bias1, float bias2, float inv_total, long long timeout_cycles, u64 cta_counter,
             int upload_dtype, int grid, u64 stream, bool dynamic_weights, float my_weight, uint32_t reducer_mask, long long shadow_skip_lo,
             long long shadow_skip_hi) {
              FedAvgParams p;
              p.shadow_skip_lo = shadow_skip_lo; p.shadow_skip_hi = shadow_skip_hi;
              p.dynamic_weights = dynamic_weights ? 1 : 0; p.my_weight = my_weight;
              p.reducer_mask = reducer_mask ? reducer_mask : ((n_reducers >= 32) ? 0xffffffffu : ((1u << n_reducers) - 1u));
              p.upload = table(upload); p.param_out = table(param_out); p.shadow_out = table(shadow_out); p.pads = table(pads);
              p.upload_mc = P<void>(upload_mc); p.param_mc = P<void>(param_mc); p.shadow_mc = P<void>(shadow_mc);
              p.w_global = P<float>(w_global); p.opt_m = P<float>(opt_m); p.opt_v = P<float>(opt_v);
              for (int i = 0; i < V6_MAX_PEERS; ++i) p.weight[i] = i < (int)weight.size() ? weight[i] : 0.f;
              p.lo = lo; p.hi = hi; p.rank = rank; p.world = world; p.n_reducers = n_reducers; p.live_mask = live_mask; p.epoch = epoch;
              p.upload_is_delta = upload_is_delta; p.upload_prescaled = upload_prescaled; p.server_opt = server_opt;
              p.server_lr = server_lr; p.beta1 = beta1; p.beta2 = beta2; p.eps = eps; p.bias1 = bias1; p.bias2 = bias2;
              p.inv_total = inv_total; p.timeout_cycles = timeout_cycles; p.cta_counter = P<unsigned int>(cta_counter);
              check(v6_fedavg_round(&p, upload_dtype, grid, S(stream)), "fedavg_round");
          });
    m.def("symm_barrier", [](const std::vector<u64>& pads, int rank, int world, uint32_t epoch, long long timeout_cycles, u64 stream) {
        PeerTable t = table(pads);
        check(v6_symm_barrier(&t, rank, world, epoch, timeout_cycles, S(stream)), "symm_barrier");
    });
    m.def("small_allreduce", [](const std::vector<u64>& slots, const std::vector<u64>& pads, const std::vector<float>& weight,
                                u64 out, int n, int rank, int world, uint32_t epoch, float inv_total, long long timeout_cycles,
                                u64 stream) {
        SmallParams p;
        p.slots = table(slots); p.pads = table(pads);
        for (int i = 0; i < V6_MAX_PEERS; ++i) p.weight[i] = i < (int)weight.size() ? weight[i] : 0.f;
        p.out = P<float>(out); p.n = n; p.rank = rank; p.world = world; p.epoch = epoch; p.inv_total = inv_total;
        p.timeout_cycles = timeout_cycles;
        check(v6_small_allreduce(&p, S(stream)), "small_allreduce");
    });
    m.def("glm_aggregate_update", [](const std::vector<u64>& slots, const std::vector<u64>& pads, const std::vector<float>& weight,
                                     u64 out, int n, int rank, int world, uint32_t epoch, long long timeout_cycles, u64 part,
                                     int nparts, int F, float rows, float lr, u64 w, u64 loss_out, u64 stream) {
        SmallParams p;
        p.slots = table(slots); p.pads = table(pads);
        for (int i = 0; i < V6_MAX_PEERS; ++i) p.weight[i] = i < (int)weight.size() ? weight[i] : 0.f;
        p.out = P<float>(out); p.n = n; p.rank = rank; p.world = world; p.epoch = epoch; p.inv_total = 1.f;
        p.timeout_cycles = timeout_cycles;
        check(v6_glm_aggregate_update(&p, P<float>(part), nparts, F, rows, lr, P<float>(w), P<float>(loss_out), S(stream)),
              "glm_aggregate_update");
    });
    m.def("p2p_pull", [](u64 src, u64 dst, long long nbytes, u64 s) { check(v6_p2p_pull(P<void>(src), P<void>(dst), nbytes, S(s)), "p2p_pull"); });
    m.def("mc_push", [](u64 src, u64 mc, long long nbytes, u64 s) { check(v6_mc_push(P<void>(src), P<void>(mc), nbytes, S(s)), "mc_push"); });
    m.def("mc_reduce", [](u64 mc, u64 dst, long long nbytes, u64 s) { check(v6_mc_reduce(P<void>(mc), P<void>(dst), nbytes, S(s)), "mc_reduce"); });

    // ------------------------------------------------------------------ K7 optimizers
    m.def("flat_optim",
          [](int kind, u64 w, u64 g, u64 mm, u64 v, u64 w_ref, u64 upload, u64 shadow, u64 grad_scale_ptr, long long n,
             float lr, float momentum, float dampening, float weight_decay, float beta1, float beta2, float eps, float bias1,
             float bias2, float contrib_scale, bool nesterov, bool save_ref, int publish, bool first_momentum_step, u64 stream,
             u64 bias_ptr, u64 contrib_scale_ptr) {
              OptimParams p;
              p.contrib_scale_ptr = P<float>(contrib_scale_ptr);
              p.w = P<float>(w); p.g = P<float>(g); p.m = P<float>(mm); p.v = P<float>(v); p.w_ref = P<float>(w_ref);
              p.upload = P<void>(upload); p.shadow = P<void>(shadow); p.grad_scale_ptr = P<float>(grad_scale_ptr); p.n = n;
              p.lr = lr; p.momentum = momentum; p.dampening = dampening; p.weight_decay = weight_decay; p.beta1 = beta1;
              p.beta2 = beta2; p.eps = eps; p.bias1 = bias1; p.bias2 = bias2; p.contrib_scale = contrib_scale;
              p.bias_ptr = P<float>(bias_ptr);
              p.nesterov = nesterov; p.save_ref = save_ref; p.publish = publish; p.first_momentum_step = first_momentum_step;
              check(kind == 0 ? v6_flat_sgd(&p, S(stream)) : v6_flat_adamw(&p, S(stream)), "flat_optim");
          });
    m.def("adam_bias_update", [](u64 step, float beta1, float beta2, u64 out, u64 s) {
        check(v6_adam_bias_update(P<int>(step), beta1, beta2, P<float>(out), S(s)), "adam_bias_update");
    });
    m.def("delta_publish", [](u64 w, u64 ref, u64 upload, long long n, float scale, bool bf16_out, u64 s) {
        check(v6_delta_publish(P<float>(w), P<float>(ref), P<void>(upload), n, scale, bf16_out, S(s)), "delta_publish");
    });
    m.def("cast_bf16", [](u64 src, u64 dst, long long n, u64 s) { check(v6_cast_bf16(P<float>(src), P<void>(dst), n, S(s)), "cast_bf16"); });
    m.def("clip_coef", [](u64 g, long long n, float max_norm, u64 scratch, u64 coef, u64 s) {
        check(v6_clip_coef(P<float>(g), n, max_norm, P<float>(scratch), P<float>(coef), S(s)), "clip_coef");
    });

    // ------------------------------------------------------------------ K5 norms
    m.def("layernorm_fwd", [](u64 x, u64 res, u64 gamma, u64 beta, u64 y, u64 res_out, u64 mean, u64 rstd, int rows, int cols,
                              float eps, bool bf16, u64 s) {
        check(v6_layernorm_fwd(P<void>(x), P<void>(res), P<float>(gamma), P<float>(beta), P<void>(y), P<void>(res_out),
                               P<float>(mean), P<float>(rstd), rows, cols, eps, bf16, S(s)), "layernorm_fwd");
    });
    m.def("rmsnorm_fwd", [](u64 x, u64 res, u64 gamma, u64 y, u64 res_out, u64 rstd, int rows, int cols, float eps, bool bf16, u64 s) {
        check(v6_rmsnorm_fwd(P<void>(x), P<void>(res), P<float>(gamma), P<void>(y), P<void>(res_out), P<float>(rstd), rows, cols,
                             eps, bf16, S(s)), "rmsnorm_fwd");
    });
    m.def("layernorm_bwd", [](u64 dy, u64 x_in, u64 dres, u64 gamma, u64 mean, u64 rstd, u64 dx, u64 dgamma, u64 dbeta,
                              u64 scratch, int parts, int rows, int cols, bool accumulate, bool bf16, u64 s) {
        check(v6_layernorm_bwd(P<void>(dy), P<void>(x_in), P<void>(dres), P<float>(gamma), P<float>(mean), P<float>(rstd),
                               P<void>(dx), P<float>(dgamma), P<float>(dbeta), P<float>(scratch), parts, rows, cols, accumulate,
                               bf16, S(s)), "layernorm_bwd");
    });
    m.def("rmsnorm_bwd", [](u64 dy, u64 x_in, u64 dres, u64 gamma, u64 rstd, u64 dx, u64 dgamma, u64 scratch, int parts,
                            int rows, int cols, bool accumulate, bool bf16, u64 s) {
        check(v6_rmsnorm_bwd(P<void>(dy), P<void>(x_in), P<void>(dres), P<float>(gamma), P<float>(rstd), P<void>(dx),
                             P<float>(dgamma), P<float>(scratch), parts, rows, cols, accumulate, bf16, S(s)), "rmsnorm_bwd");
    });

    // ------------------------------------------------------------------ fused BatchNorm (+add)(+ReLU), NHWC bf16
    m.def("multi_accum_bf16", [](std::vector<u64> src, std::vector<long long> off, std::vector<long long> numel, u64 dst, u64 s) {
        if (src.size() != off.size() || src.size() != numel.size()) throw std::runtime_error("multi_accum_bf16: list sizes differ");
        for (size_t base = 0; base < src.size(); base += V6_MULTI_MAX) {
            MultiAccumParams p;
            p.count = (int)std::min<size_t>(V6_MULTI_MAX, src.size() - base);
            for (int i = 0; i < p.count; ++i) {
                p.src[i] = P<void>(src[base + i]);
                p.dst_off[i] = off[base + i];
                p.numel[i] = numel[base + i];
            }
            check(v6_multi_accum_bf16(&p, P<float>(dst), S(s)), "multi_accum_bf16");
        }
    });
    m.def("maxpool3x3s2_fwd", [](u64 x, u64 y, u64 idx, int N, int H, int W, int C, u64 s) {
        check(v6_maxpool3x3s2_fwd(P<void>(x), P<void>(y), P<void>(idx), N, H, W, C, S(s)), "maxpool3x3s2_fwd");
    });
    m.def("maxpool3x3s2_bwd", [](u64 dy, u64 idx, u64 dx, int N, int H, int W, int C, u64 s) {
        check(v6_maxpool3x3s2_bwd(P<void>(dy), P<void>(idx), P<void>(dx), N, H, W, C, S(s)), "maxpool3x3s2_bwd");
    });
    m.def("image_normalize", [](u64 img, u64 out, long long N, long long HW, float m0, float m1, float m2, float s0, float s1,
                                float s2, u64 s) {
        check(v6_image_normalize(P<void>(img), P<void>(out), N, HW, m0, m1, m2, s0, s1, s2, S(s)), "image_normalize");
    });
    m.def("image_normalize_s2d", [](u64 img, u64 out, int N, int H, int W, float m0, float m1, float m2, float s0, float s1, float s2,
                                    u64 s) {
        check(v6_image_normalize_s2d(P<void>(img), P<void>(out), N, H, W, m0, m1, m2, s0, s1, s2, S(s)), "image_normalize_s2d");
    });
    m.def("stem_weight_s2d", [](u64 w, bool w_is_bf16, u64 ws, int O, u64 s) {
        check(v6_stem_weight_s2d(P<void>(w), w_is_bf16, P<void>(ws), O, S(s)), "stem_weight_s2d");
    });
    m.def("stem_wgrad_d2s", [](u64 dws, u64 dw, int O, bool accumulate, u64 s) {
        check(v6_stem_wgrad_d2s(P<void>(dws), P<float>(dw), O, accumulate, S(s)), "stem_wgrad_d2s");
    });
    m.def("bias_act_bwd", [](u64 dy, u64 pre, u64 dpre, u64 db, u64 scratch, long long R, int C, int act, bool accumulate, u64 s) {
        check(v6_bias_act_bwd(P<void>(dy), P<void>(pre), P<void>(dpre), P<float>(db), P<float>(scratch), R, C, act, accumulate, S(s)),
              "bias_act_bwd");
    });
    m.def("swiglu_fwd", [](u64 g, u64 u, u64 h, long long n, u64 s) {
        check(v6_swiglu_fwd(P<void>(g), P<void>(u), P<void>(h), n, S(s)), "swiglu_fwd");
    });
    m.def("swiglu_bwd", [](u64 dh, u64 g, u64 u, u64 dg, u64 du, long long n, u64 s) {
        check(v6_swiglu_bwd(P<void>(dh), P<void>(g), P<void>(u), P<void>(dg), P<void>(du), n, S(s)), "swiglu_bwd");
    });
    m.def("bn_fwd", [](u64 x, u64 res, u64 gamma, u64 beta, u64 rmean, u64 rvar, u64 nbt, u64 y, u64 mask, u64 mean, u64 rstd,
                       u64 scale_bias, u64 scratch, long long R, int C, float eps, float momentum, bool relu, u64 s) {
        check(v6_bn_fwd(P<void>(x), P<void>(res), P<float>(gamma), P<float>(beta), P<float>(rmean), P<float>(rvar),
                        P<long long>(nbt), P<void>(y), P<void>(mask), P<float>(mean), P<float>(rstd), P<float>(scale_bias), P<float>(scratch), R,
                        C, eps, momentum, relu, S(s)),
              "bn_fwd");
    });
    m.def("bn_apply", [](u64 x, u64 res, u64 scale, u64 bias, u64 y, u64 mask, long long R, int C, bool relu, u64 s) {
        check(v6_bn_apply(P<void>(x), P<void>(res), P<float>(scale), P<float>(bias), P<void>(y), P<void>(mask), R, C, relu, S(s)), "bn_apply");
    });
    m.def("bn_bwd", [](u64 dy, u64 y, u64 x, u64 gamma, u64 mean, u64 rstd, u64 dx, u64 dres, u64 dgamma, u64 dbeta, u64 coef,
                       u64 scratch, long long R, int C, bool relu, bool accumulate, u64 s) {
        check(v6_bn_bwd(P<void>(dy), P<void>(y), P<void>(x), P<float>(gamma), P<float>(mean), P<float>(rstd), P<void>(dx),
                        P<void>(dres), P<float>(dgamma), P<float>(dbeta), P<float>(coef), P<float>(scratch), R, C, relu,
                        accumulate, S(s)), "bn_bwd");
    });
    m.def("ce_fwd", [](u64 logits, u64 labels, u64 lse, u64 loss, int T, int V, long long ld, long long ignore_index, u64 s) {
        check(v6_ce_fwd(P<void>(logits), P<long long>(labels), P<float>(lse), P<float>(loss), T, V, ld, ignore_index, S(s)), "ce_fwd");
    });
    m.def("ce_bwd", [](u64 logits, u64 labels, u64 lse, u64 scale, int T, int V, int V_alloc, long long ld, long long ignore_index, u64 s) {
        check(v6_ce_bwd(P<void>(logits), P<long long>(labels), P<float>(lse), P<float>(scale), T, V, V_alloc, ld, ignore_index, S(s)), "ce_bwd");
    });
    m.attr("BN_SCRATCH_FLOATS") = v6_bn_scratch_floats();

    // ------------------------------------------------------------------ K6 / K8
    m.def("rope", [](u64 q, u64 k, u64 cos_t, u64 sin_t, u64 pos, int B, int Sq, int Hq, int Hkv, int D, bool inverse, u64 s) {
        check(v6_rope(P<void>(q), P<void>(k), P<float>(cos_t), P<float>(sin_t), P<int>(pos), B, Sq, Hq, Hkv, D, inverse, S(s)), "rope");
    });
    m.def("glm_logistic_partials_tc", [](u64 X, u64 y, u64 w, u64 part, int max_parts, int rows, int F, u64 s) {
        const int grid = v6_glm_logistic_grad_tc(P<void>(X), P<float>(y), P<float>(w), P<float>(part), max_parts, rows, F, S(s));
        if (grid < 1) throw std::runtime_error("glm_logistic_partials_tc failed (" + std::to_string(grid) + ")");
        return grid;
    });
    m.def("glm_logistic_grad_tc", [](u64 X, u64 y, u64 w, u64 part, int max_parts, u64 out, int rows, int F, u64 s) {
        const int grid = v6_glm_logistic_grad_tc(P<void>(X), P<float>(y), P<float>(w), P<float>(part), max_parts, rows, F, S(s));
        if (grid < 1) throw std::runtime_error("glm_logistic_grad_tc failed (" + std::to_string(grid) + ")");
        check(v6_glm_fold(P<float>(part), P<float>(out), grid, F, rows, S(s)), "glm_fold");
    });
    m.def("glm_logistic_grad", [](u64 X, u64 y, u64 w, u64 part, int max_parts, u64 out, int rows, int F, bool bf16, u64 s) {
        check(v6_glm_logistic_grad(P<void>(X), P<float>(y), P<float>(w), P<float>(part), max_parts, P<float>(out), rows, F, bf16, S(s)),
              "glm_logistic_grad");
    });

    // ------------------------------------------------------------------ implicit-GEMM convolution family (igemm.cu)
    m.attr("IGEMM_SCRATCH_FLOATS") = v6_igemm_scratch_floats();
    m.def("stem_wgrad_d2s_f32", [](u64 dws, u64 dw, int O, bool accumulate, u64 s) {
        check(v6_stem_wgrad_d2s_f32(P<float>(dws), P<float>(dw), O, accumulate, S(s)), "stem_wgrad_d2s_f32");
    });
    m.def("conv_fprop", [](u64 x, u64 w, u64 y, u64 bias, int act, int N, int H, int W, int Cin, int Cout, int R, int Sw, int stride,
                           int pad, u64 gamma, u64 beta, u64 rmean, u64 rvar, u64 nbt, u64 mean, u64 rstd, u64 scale_bias,
                           u64 scratch, float eps, float momentum, bool force_im2col, u64 s, long long pitch_w, long long pitch_h,
                           long long pitch_n) {
        check(v6_conv_fprop(P<void>(x), P<void>(w), P<void>(y), P<float>(bias), act, N, H, W, Cin, Cout, R, Sw, stride, pad,
                            P<float>(gamma), P<float>(beta), P<float>(rmean), P<float>(rvar), P<long long>(nbt), P<float>(mean),
                            P<float>(rstd), P<float>(scale_bias), P<float>(scratch), eps, momentum, force_im2col, pitch_w, pitch_h,
                            pitch_n, S(s)),
              "conv_fprop");
    });
    m.def("conv_dgrad", [](u64 dy, u64 w, u64 dx, int N, int H, int W, int Cin, int Cout, int R, int Sw, int stride, int pad,
                           bool force_im2col, u64 s, u64 add_src, u64 add_mask) {
        check(v6_conv_dgrad(P<void>(dy), P<void>(w), P<void>(dx), N, H, W, Cin, Cout, R, Sw, stride, pad, force_im2col, P<void>(add_src), P<void>(add_mask),
                            S(s)), "conv_dgrad");
    });
    m.def("conv_wgrad", [](u64 dy, u64 x, u64 dw, int N, int H, int W, int Cin, int Cout, int R, int Sw, int stride, int pad,
                           float scale, int splits, bool force_im2col, u64 s, long long pitch_w, long long pitch_h, long long pitch_n,
                           u64 ws, long long ws_floats) {
        check(v6_conv_wgrad(P<void>(dy), P<void>(x), P<float>(dw), N, H, W, Cin, Cout, R, Sw, stride, pad, scale, splits,
                            force_im2col, pitch_w, pitch_h, pitch_n, P<float>(ws), ws_floats, S(s)), "conv_wgrad");
    });
    m.def("conv_wgrad_workspace", &v6_conv_wgrad_workspace);
    // ------------------------------------------------------------------ K1 / tcgen05 GEMM
    m.def("gemm_bf16", [](u64 A, u64 B, u64 C, u64 bias, int M, int N, int K, int lda, int ldb, int ldc, int act, u64 s) {
        check(v6_gemm_bf16(P<void>(A), P<void>(B), P<void>(C), P<float>(bias), M, N, K, lda, ldb, ldc, act, S(s)), "gemm_bf16");
    });
    m.def("gemm2_bf16", [](u64 A, u64 B, u64 C, u64 bias, int M, int N, int K, int lda, int ldb, int ldc, int act, u64 s) {
        check(v6_gemm2_bf16(P<void>(A), P<void>(B), P<void>(C), P<float>(bias), M, N, K, lda, ldb, ldc, act, S(s)), "gemm2_bf16");
    });
    m.def("bcast_gemm_bf16", [](u64 A, u64 B_local, u64 B_peer, u64 C, u64 bias, int M, int N, int K, int lda, int ldb, int ldc,
                                int act, u64 flags, uint32_t epoch, u64 s) {
        check(v6_bcast_gemm_bf16(P<void>(A), P<void>(B_local), P<void>(B_peer), P<void>(C), P<float>(bias), M, N, K, lda, ldb,
                                 ldc, act, P<uint32_t>(flags), epoch, S(s)), "bcast_gemm_bf16");
    });
    m.def("gemm_smem_bytes", &v6_gemm_smem_bytes);
    m.def("bcast_push_gemm_bf16", [](u64 A, u64 B_local, u64 B_mc, u64 C, u64 bias, int M, int N, int K, int lda, int ldb, int ldc,
                                     int act, u64 flags, const std::vector<u64>& flag_peers, int world, bool is_owner, uint32_t epoch,
                                     u64 s, int own_nb_lo, int own_nb_hi, u64 epoch_ptr, u64 status_ptr) {
        PeerTable t = table(flag_peers);
        check(v6_bcast_push_gemm_bf16(P<void>(A), P<void>(B_local), P<void>(B_mc), P<void>(C), P<float>(bias), M, N, K, lda, ldb,
                                      ldc, act, P<uint32_t>(flags), &t, world, is_owner ? 1 : 0, epoch, own_nb_lo, own_nb_hi,
                                      P<uint32_t>(epoch_ptr), P<uint32_t>(status_ptr), S(s)), "bcast_push_gemm_bf16");
    });

    m.def("flash_attn_bwd", [](u64 q, u64 k, u64 v, u64 dout, u64 kt, u64 qt, u64 dot, u64 lse2, u64 delta, u64 dq, u64 dk,
                               u64 dv, int B, int Sq, int Hq, int Hkv, int D, float scale, bool causal, u64 s) {
        check(v6_flash_attn_bwd(P<void>(q), P<void>(k), P<void>(v), P<void>(dout), P<void>(kt), P<void>(qt), P<void>(dot),
                                P<float>(lse2), P<float>(delta), P<void>(dq), P<void>(dk), P<void>(dv), B, Sq, Hq, Hkv, D,
                                scale, causal, S(s)), "flash_attn_bwd");
    });
    // ------------------------------------------------------------------ K4 attention
    m.def("flash_attn_fwd2_vmn", [](u64 q, u64 k, u64 v, u64 o, u64 lse, int B, int Sq, int Hq, int Hkv, int D, long long ldq,
                                   long long ldk, long long ldv, float scale, bool causal, u64 s) {
        check(v6_flash_attn_fwd2_vmn(P<void>(q), P<void>(k), P<void>(v), P<void>(o), P<float>(lse), B, Sq, Hq, Hkv, D, ldq, ldk, ldv,
                                     scale, causal, S(s)), "flash_attn_fwd2_vmn");
    });
    m.def("flash_attn_fwd2", [](u64 q, u64 k, u64 vt, u64 o, u64 lse, int B, int Sq, int Hq, int Hkv, int D, long long ldq, long long ldk, float scale,
                               bool causal, u64 s) {
        check(v6_flash_attn_fwd2(P<void>(q), P<void>(k), P<void>(vt), P<void>(o), P<float>(lse), B, Sq, Hq, Hkv, D, ldq, ldk, scale,
                                 causal, S(s)), "flash_attn_fwd2");
    });
    m.def("flash_attn_fwd", [](u64 q, u64 k, u64 vt, u64 o, u64 lse, int B, int Sq, int Hq, int Hkv, int D, long long ldq, long long ldk, float scale,
                               bool causal, u64 s) {
        check(v6_flash_attn_fwd(P<void>(q), P<void>(k), P<void>(vt), P<void>(o), P<float>(lse), B, Sq, Hq, Hkv, D, ldq, ldk, scale,
                                causal, S(s)), "flash_attn_fwd");
    });
}
