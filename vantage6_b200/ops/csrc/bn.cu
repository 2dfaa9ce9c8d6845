// Fused BatchNorm(+residual add)(+ReLU) forward / backward for NHWC bf16 activations (ResNet-50).
//
// The first profile of the flagship local step (profiles/launches_resnet50_eager_r1.txt) showed
// PyTorch's native channels-last BatchNorm kernels + stand-alone ReLU / add kernels taking ~3/4 of
// the GPU time of a ResNet-50 step on B200 -- the convolutions (cuDNN/CUTLASS sm100 kernels) only
// ~15%.  These kernels make that part memory-bound at HBM speed and remove the separate ReLU /
// residual-add passes:
//
//   forward :  stats + per-channel finalize (1 read of x, one launch)  ->  y = relu(x*scale + bias + res)
//   backward:  reduce + finalize (dy, y, x -> dgamma, dbeta, coefficients)  ->  dx (and dres) in one pass
//
// x viewed as [R = N*H*W, C], C % 8 == 0 and C/8 a power of two <= 256 (64..2048 in ResNet-50).
// Element-wise passes: threadIdx % (C/8) owns 8 consecutive channels (one 16 B vector), threadIdx / (C/8)
// is a row lane; CTAs stride over rows.  Reductions: see "in-kernel tree reduction" below; per-channel
// sums are accumulated in registers across rows (shifted by x[0,c] to avoid cancellation in
// E[x^2]-E[x]^2) -- no floating-point atomics, deterministic.
#include "common.cuh"
#include "api.h"
#include "tree_reduce.cuh"

namespace bn {

using namespace tree;          // THREADS, Red, slice_reduce, reduce_grid, wave_ctas (tree_reduce.cuh)

// Programmatic dependent launch (PDL): the element-wise pass of a BN layer is launched with
// cudaLaunchAttributeProgrammaticStreamSerialization, so its CTAs are scheduled while the reduction kernel's tree
// tail is still running and block in griddepcontrol.wait until that grid has completed and flushed its writes.
// Without the attribute both instructions are no-ops.
V6_DEVINL void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
V6_DEVINL void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

V6_DEVINL void load8(const __nv_bfloat16* p, float (&v)[8]) {
    uint4 t = *reinterpret_cast<const uint4*>(p);
    float2 a = unpack_bf16x2(t.x), b = unpack_bf16x2(t.y), c = unpack_bf16x2(t.z), d = unpack_bf16x2(t.w);
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; v[4] = c.x; v[5] = c.y; v[6] = d.x; v[7] = d.y;
}
V6_DEVINL void store8(__nv_bfloat16* p, const float (&v)[8]) {
    *reinterpret_cast<uint4*>(p) = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]),
                                              pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
}
V6_DEVINL uint4 ldg_nc_v4(const __nv_bfloat16* p) { return __ldg(reinterpret_cast<const uint4*>(p)); }
V6_DEVINL void unpack8(const uint4& t, float (&v)[8]) {
    float2 a = unpack_bf16x2(t.x), b = unpack_bf16x2(t.y), c = unpack_bf16x2(t.z), d = unpack_bf16x2(t.w);
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; v[4] = c.x; v[5] = c.y; v[6] = d.x; v[7] = d.y;
}
V6_DEVINL void acc_stats(const uint4& raw, const float (&shift)[8], float (&s1)[8], float (&s2)[8]) {
    float v[8];
    unpack8(raw, v);
#pragma unroll
    for (int k = 0; k < 8; ++k) { const float d = v[k] - shift[k]; s1[k] += d; s2[k] = fmaf(d, d, s2[k]); }
}
V6_DEVINL void loadf8(const float* p, float (&v)[8]) {
    float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}

// ---------------------------------------------------------------------------------- forward
// stats + finalize: per-channel mean / rstd / (scale, bias) of y = x*scale + bias, running-stat update.
constexpr int STATS_UNROLL = 4;
__global__ void __launch_bounds__(THREADS, 4) bn_stats_kernel(const __nv_bfloat16* __restrict__ x, Red rd,
                                       const float* __restrict__ gamma, const float* __restrict__ beta,
                                       float* __restrict__ running_mean, float* __restrict__ running_var,
                                       long long* __restrict__ num_batches_tracked,
                                       float* __restrict__ mean_out, float* __restrict__ rstd_out,
                                       float* __restrict__ scale_out, float* __restrict__ bias_out,
                                       long long R, int C, float eps, float momentum) {
    __shared__ float tot[128];
    const int SW = C < 64 ? C : 64, CGS = SW >> 3, RL = THREADS / CGS;
    const int cg = threadIdx.x % CGS, rl = threadIdx.x / CGS;
    const __nv_bfloat16* xc = x + blockIdx.y * SW + cg * 8;
    float shift[8], s1[8], s2[8];
    load8(xc, shift);                                           // row 0 as the per-channel shift
#pragma unroll
    for (int k = 0; k < 8; ++k) { s1[k] = 0.f; s2[k] = 0.f; }
    const long long G = (long long)gridDim.x * RL;
    long long r = (long long)blockIdx.x * RL + rl;
    for (; r + (STATS_UNROLL - 1) * G < R; r += STATS_UNROLL * G) {            // UNROLL independent 16 B loads in flight
        uint4 raw[STATS_UNROLL];
#pragma unroll
        for (int u = 0; u < STATS_UNROLL; ++u) raw[u] = ldg_nc_v4(xc + (r + u * G) * C);
#pragma unroll
        for (int u = 0; u < STATS_UNROLL; ++u) acc_stats(raw[u], shift, s1, s2);
    }
    for (; r < R; r += G) acc_stats(ldg_nc_v4(xc + r * C), shift, s1, s2);
    pdl_launch_dependents();                                   // let the apply kernel's CTAs get scheduled
    if (!slice_reduce(s1, s2, rd, SW, tot)) return;
    if (threadIdx.x < SW) {
        const int c = blockIdx.y * SW + threadIdx.x;
        const float sh = __bfloat162float(x[c]);
        const float invR = 1.f / (float)R;
        const float dm = tot[threadIdx.x] * invR;
        const float mean = sh + dm;
        const float var = fmaxf(tot[SW + threadIdx.x] * invR - dm * dm, 0.f);
        const float rstd = rsqrtf(var + eps);
        mean_out[c] = mean;
        rstd_out[c] = rstd;
        const float sc = gamma[c] * rstd;
        scale_out[c] = sc;
        bias_out[c] = beta[c] - mean * sc;
        if (running_mean) {
            const float unbiased = R > 1 ? var * (float)R / (float)(R - 1) : var;
            running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * mean;
            running_var[c] = (1.f - momentum) * running_var[c] + momentum * unbiased;
        }
        if (num_batches_tracked && c == 0) *num_batches_tracked += 1;
    }
}

// Element-wise passes: U rows per thread are requested (raw 16 B vectors, kept packed until used) before the first one
// is consumed, and the grid is exactly one wave of resident CTAs (apply_grid) -- HBM3e wants >= ~64 KB of loads in flight
// per SM and a grid-stride loop has no tail.  Launched with U = 2 at 3 CTAs/SM, coefficients in registers:
// 2.52 ms of these passes per ResNet-50 step on a B200, vs 2.93 ms with U = 4 at 4 CTAs/SM (coefficients in shared memory) and 2.51 ms with U = 4 at 2 CTAs/SM (profiles/bn_bench_r2f.jsonl).
template <bool RELU, bool RES, int U, int MINB>
__global__ void __launch_bounds__(THREADS, MINB) bn_apply_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ res,
                                                                 const float* __restrict__ scale, const float* __restrict__ bias,
                                                                 __nv_bfloat16* __restrict__ y, unsigned char* __restrict__ mask,
                                                                 long long R, int C) {
    const int CG = C >> 3, RL = THREADS / CG;
    const int cg = threadIdx.x % CG, rl = threadIdx.x / CG;
    pdl_wait();                                                 // scale / bias come from the stats kernel
    float sc[8], bi[8];
    loadf8(scale + cg * 8, sc);
    loadf8(bias + cg * 8, bi);
    const long long G = (long long)gridDim.x * RL;
    for (long long r0 = (long long)blockIdx.x * RL + rl; r0 < R; r0 += U * G) {
        uint4 xr[U], qr[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const long long r = r0 + u * G;
            if (r < R) {
                xr[u] = ldg_nc_v4(x + r * C + cg * 8);
                if (RES) qr[u] = ldg_nc_v4(res + r * C + cg * 8);
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const long long r = r0 + u * G;
            if (r < R) {
                float v[8], q[8];
                unpack8(xr[u], v);
                if (RES) unpack8(qr[u], q);
                unsigned bits = 0;
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    float t = fmaf(v[k], sc[k], bi[k]);
                    if (RES) t += q[k];
                    if (RELU) bits |= (t > 0.f ? 1u : 0u) << k;
                    v[k] = RELU ? fmaxf(t, 0.f) : t;
                }
                store8(y + r * C + cg * 8, v);
                if (RELU && mask) mask[r * CG + cg] = (unsigned char)bits;      // 1 bit / element for the backward
            }
        }
    }
}

// ---------------------------------------------------------------------------------- backward
template <bool RELU>
V6_DEVINL void acc_bwd(const uint4& graw, const uint4& xraw, unsigned bits, const float (&mu)[8], const float (&rs)[8],
                       float (&sg)[8], float (&sgx)[8]) {
    float g[8], xv[8];
    unpack8(graw, g);
    unpack8(xraw, xv);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const float gg = (RELU && !((bits >> k) & 1u)) ? 0.f : g[k];
        sg[k] += gg;
        sgx[k] = fmaf(gg, (xv[k] - mu[k]) * rs[k], sgx[k]);
    }
}

// reduce + finalize: per channel dgamma, dbeta (optionally accumulated into the flat fp32 grad buffer) and
// the coefficients of dx = c0 * g + c1 * x + c2 with
//   c0 = gamma*rstd, c1 = -gamma*rstd^2*mean(g*xhat), c2 = -c0*mean(g) - c1*mean
constexpr int RED_UNROLL = 4;
template <bool RELU>
__global__ void __launch_bounds__(THREADS, 3) bn_bwd_reduce_kernel(const __nv_bfloat16* __restrict__ dy, const unsigned char* __restrict__ mask,
                                       const __nv_bfloat16* __restrict__ x, const float* __restrict__ gamma,
                                       const float* __restrict__ mean, const float* __restrict__ rstd, Red rd,
                                       float* __restrict__ dgamma, float* __restrict__ dbeta, float* __restrict__ coef,
                                       long long R, int C, int accumulate) {
    __shared__ float tot[128];
    const int SW = C < 64 ? C : 64, CGS = SW >> 3, RL = THREADS / CGS;
    const int cg = threadIdx.x % CGS, rl = threadIdx.x / CGS;
    const size_t c0 = (size_t)blockIdx.y * SW + cg * 8;
    pdl_wait();                                                 // dy comes from the kernel before (programmatic dependent launch)
    const long long CGT = C >> 3, cgt = (long long)blockIdx.y * CGS + cg;       // mask: [R][C/8] bytes
    float mu[8], rs[8], sg[8], sgx[8];
    loadf8(mean + c0, mu);
    loadf8(rstd + c0, rs);
#pragma unroll
    for (int k = 0; k < 8; ++k) { sg[k] = 0.f; sgx[k] = 0.f; }
    const long long G = (long long)gridDim.x * RL;
    long long r = (long long)blockIdx.x * RL + rl;
    for (; r + (RED_UNROLL - 1) * G < R; r += RED_UNROLL * G) {                // RED_UNROLL rows x 3 tensors in flight
        uint4 g[RED_UNROLL], xv[RED_UNROLL];
        unsigned mb[RED_UNROLL];
#pragma unroll
        for (int u = 0; u < RED_UNROLL; ++u) {
            const long long o = (r + u * G) * C + c0;
            g[u] = ldg_nc_v4(dy + o);
            xv[u] = ldg_nc_v4(x + o);
            mb[u] = RELU ? (unsigned)__ldg(mask + (r + u * G) * CGT + cgt) : 0xffu;
        }
#pragma unroll
        for (int u = 0; u < RED_UNROLL; ++u) acc_bwd<RELU>(g[u], xv[u], mb[u], mu, rs, sg, sgx);
    }
    for (; r < R; r += G) {
        const long long o = r * C + c0;
        unsigned mb = 0xffu;
        if (RELU) mb = __ldg(mask + r * CGT + cgt);
        acc_bwd<RELU>(ldg_nc_v4(dy + o), ldg_nc_v4(x + o), mb, mu, rs, sg, sgx);
    }
    pdl_launch_dependents();
    if (!slice_reduce(sg, sgx, rd, SW, tot)) return;
    if (threadIdx.x < SW) {
        const int c = blockIdx.y * SW + threadIdx.x;
        const float tg = tot[threadIdx.x], tgx = tot[SW + threadIdx.x];
        dgamma[c] = accumulate ? dgamma[c] + tgx : tgx;
        dbeta[c] = accumulate ? dbeta[c] + tg : tg;
        const float invR = 1.f / (float)R;
        const float k0 = gamma[c] * rstd[c];
        const float k1 = -k0 * rstd[c] * tgx * invR;
        coef[c] = k0;
        coef[C + c] = k1;
        coef[2 * C + c] = -k0 * tg * invR - k1 * mean[c];
    }
}

template <bool RELU, bool RES, int U, int MINB>
__global__ void __launch_bounds__(THREADS, MINB) bn_bwd_apply_kernel(const __nv_bfloat16* __restrict__ dy, const unsigned char* __restrict__ mask,
                                                                     const __nv_bfloat16* __restrict__ x, const float* __restrict__ coef,
                                                                     __nv_bfloat16* __restrict__ dx, __nv_bfloat16* __restrict__ dres,
                                                                     long long R, int C) {
    const int CG = C >> 3, RL = THREADS / CG;
    const int cg = threadIdx.x % CG, rl = threadIdx.x / CG;
    pdl_wait();                                                 // coefficients come from the reduce kernel
    float c0[8], c1[8], c2[8];
    loadf8(coef + cg * 8, c0);
    loadf8(coef + C + cg * 8, c1);
    loadf8(coef + 2 * C + cg * 8, c2);
    const long long G = (long long)gridDim.x * RL;
    for (long long r0 = (long long)blockIdx.x * RL + rl; r0 < R; r0 += U * G) {
        uint4 gr[U], xr[U];
        unsigned mb[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const long long r = r0 + u * G;
            mb[u] = 0xffu;
            if (r < R) {
                gr[u] = ldg_nc_v4(dy + r * C + cg * 8);
                xr[u] = ldg_nc_v4(x + r * C + cg * 8);
                if (RELU) mb[u] = __ldg(mask + r * CG + cg);
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const long long r = r0 + u * G;
            if (r < R) {
                float g[8], xv[8], o[8];
                unpack8(gr[u], g);
                unpack8(xr[u], xv);
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    if (RELU && !((mb[u] >> k) & 1u)) g[k] = 0.f;
                    o[k] = fmaf(c0[k], g[k], fmaf(c1[k], xv[k], c2[k]));
                }
                if (RES) store8(dres + r * C + cg * 8, g);
                store8(dx + r * C + cg * 8, o);
            }
        }
    }
}

static inline bool shape_ok(int C) {
    const int cg = C >> 3;
    return C % 8 == 0 && cg >= 1 && cg <= THREADS && (cg & (cg - 1)) == 0;     // 8, 16, ..., 2048
}
// element-wise passes keep no partials: exactly one wave of resident CTAs (occupancy queried once per instantiation),
// fewer when the tensor has fewer row groups than that
template <typename K>
static int apply_grid(K kernel, long long R, int C) {
    int dev = 0, sms = 148, occ = 1;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, THREADS, 0) != cudaSuccess || occ < 1) occ = 1;
    const int RL = THREADS / (C >> 3);
    const long long g = (R + RL - 1) / RL, cap = (long long)occ * sms;
    return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

// launch `kernel` as a programmatic dependent of the previous kernel in the stream (V6B200_PDL=0 or pdl=false: plain launch)
template <typename... KArgs, typename... Args>
static void launch_dependent(void (*kernel)(KArgs...), int grid, bool dependent, cudaStream_t s, Args... args) {
    static const bool pdl = [] { const char* e = getenv("V6B200_PDL"); return !(e && e[0] == '0'); }();
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(THREADS);
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = (pdl && dependent) ? 1 : 0;
    cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// same, 2-D grid (the reduce kernels)
template <typename... KArgs, typename... Args>
static void launch_dependent_grid(void (*kernel)(KArgs...), dim3 grid, cudaStream_t s, Args... args) {
    static const bool pdl = [] { const char* e = getenv("V6B200_PDL"); return !(e && e[0] == '0'); }();
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(THREADS);
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

template <bool RELU, bool RES>
static void launch_apply(bool dependent, cudaStream_t s, const __nv_bfloat16* x, const __nv_bfloat16* res, const float* scale, const float* bias,
                         __nv_bfloat16* y, unsigned char* mask, long long R, int C) {
    auto k = bn_apply_kernel<RELU, RES, 2, 3>;
    launch_dependent(k, apply_grid(k, R, C), dependent, s, x, res, scale, bias, y, mask, R, C);
}

template <bool RELU, bool RES>
static void launch_bwd_apply(cudaStream_t s, const __nv_bfloat16* dy, const unsigned char* mask, const __nv_bfloat16* x, const float* coef,
                             __nv_bfloat16* dx, __nv_bfloat16* dres, long long R, int C) {
    auto k = bn_bwd_apply_kernel<RELU, RES, 2, 3>;
    launch_dependent(k, apply_grid(k, R, C), true, s, dy, mask, x, coef, dx, dres, R, C);
}

}  // namespace bn

// scratch: v6_bn_scratch_floats() floats, zero-initialised once (partials + self-resetting counters), shared by
// every launch on one stream.  stats: mean[C] rstd[C] scale_bias[2C].
extern "C" long long v6_bn_scratch_floats() { return (long long)tree::SCR_FLOATS; }

extern "C" int v6_bn_fwd(const void* x, const void* res, const float* gamma, const float* beta, float* running_mean,
                         float* running_var, long long* num_batches_tracked, void* y, void* relu_mask, float* mean, float* rstd,
                         float* scale_bias, float* scratch, long long R, int C, float eps, float momentum, int relu,
                         cudaStream_t s) {
    using namespace bn;
    if (!shape_ok(C)) return (int)cudaErrorInvalidValue;
    static int wave = 0;
    bn_stats_kernel<<<reduce_grid(R, C, wave_ctas(bn_stats_kernel, wave)), THREADS, 0, s>>>((const __nv_bfloat16*)x, make_red(scratch), gamma, beta,
                                                                  running_mean, running_var, num_batches_tracked, mean, rstd,
                                                                  scale_bias, scale_bias + C, R, C, eps, momentum);
    const __nv_bfloat16* xx = (const __nv_bfloat16*)x;
    const __nv_bfloat16* rr = (const __nv_bfloat16*)res;
    __nv_bfloat16* yy = (__nv_bfloat16*)y;
    unsigned char* mk = (unsigned char*)relu_mask;
    if (relu) {
        if (res) launch_apply<true, true>(true, s, xx, rr, scale_bias, scale_bias + C, yy, mk, R, C);
        else launch_apply<true, false>(true, s, xx, rr, scale_bias, scale_bias + C, yy, mk, R, C);
    } else {
        if (res) launch_apply<false, true>(true, s, xx, rr, scale_bias, scale_bias + C, yy, nullptr, R, C);
        else launch_apply<false, false>(true, s, xx, rr, scale_bias, scale_bias + C, yy, nullptr, R, C);
    }
    V6_CHECK_LAUNCH();
    return 0;
}

// inference / eval: y = relu(x*scale + bias + res) with caller-provided per-channel affine
extern "C" int v6_bn_apply(const void* x, const void* res, const float* scale, const float* bias, void* y, void* relu_mask,
                           long long R, int C, int relu, cudaStream_t s) {
    using namespace bn;
    if (!shape_ok(C)) return (int)cudaErrorInvalidValue;
    const __nv_bfloat16* xx = (const __nv_bfloat16*)x;
    const __nv_bfloat16* rr = (const __nv_bfloat16*)res;
    __nv_bfloat16* yy = (__nv_bfloat16*)y;
    unsigned char* mk = (unsigned char*)relu_mask;      // training with statistics from the convolution epilogue: 1 bit / element
    // (x and the statistics come from the convolution kernel before it, which releases its dependents at its start: this
    // kernel's CTAs are resident and past their prologue when that grid drains, and wait for it in griddepcontrol.wait)
    if (relu) {
        if (res) launch_apply<true, true>(true, s, xx, rr, scale, bias, yy, mk, R, C);
        else launch_apply<true, false>(true, s, xx, rr, scale, bias, yy, mk, R, C);
    } else {
        if (res) launch_apply<false, true>(true, s, xx, rr, scale, bias, yy, nullptr, R, C);
        else launch_apply<false, false>(true, s, xx, rr, scale, bias, yy, nullptr, R, C);
    }
    V6_CHECK_LAUNCH();
    return 0;
}

// coef scratch: 3*C floats. dres may be null (no residual branch).
extern "C" int v6_bn_bwd(const void* dy, const void* relu_mask, const void* x, const float* gamma, const float* mean, const float* rstd,
                         void* dx, void* dres, float* dgamma, float* dbeta, float* coef, float* scratch, long long R, int C,
                         int relu, int accumulate, cudaStream_t s) {
    using namespace bn;
    if (!shape_ok(C)) return (int)cudaErrorInvalidValue;
    const __nv_bfloat16* dyy = (const __nv_bfloat16*)dy;
    const unsigned char* yy = (const unsigned char*)relu_mask;     // 1 bit / element, written by the forward apply pass
    const __nv_bfloat16* xx = (const __nv_bfloat16*)x;
    if (relu && !relu_mask) return (int)cudaErrorInvalidValue;
    static int wave_relu = 0, wave_lin = 0;
    const dim3 rg = reduce_grid(R, C, relu ? wave_ctas(bn_bwd_reduce_kernel<true>, wave_relu) : wave_ctas(bn_bwd_reduce_kernel<false>, wave_lin));
    if (relu) launch_dependent_grid(bn_bwd_reduce_kernel<true>, rg, s, dyy, yy, xx, gamma, mean, rstd, make_red(scratch), dgamma, dbeta, coef, R, C, accumulate);
    else launch_dependent_grid(bn_bwd_reduce_kernel<false>, rg, s, dyy, yy, xx, gamma, mean, rstd, make_red(scratch), dgamma, dbeta, coef, R, C, accumulate);
    __nv_bfloat16* dxx = (__nv_bfloat16*)dx;
    __nv_bfloat16* drr = (__nv_bfloat16*)dres;
    if (relu) {
        if (dres) launch_bwd_apply<true, true>(s, dyy, yy, xx, coef, dxx, drr, R, C);
        else launch_bwd_apply<true, false>(s, dyy, yy, xx, coef, dxx, drr, R, C);
    } else {
        if (dres) launch_bwd_apply<false, true>(s, dyy, yy, xx, coef, dxx, drr, R, C);
        else launch_bwd_apply<false, false>(s, dyy, yy, xx, coef, dxx, drr, R, C);
    }
    V6_CHECK_LAUNCH();
    return 0;
}
