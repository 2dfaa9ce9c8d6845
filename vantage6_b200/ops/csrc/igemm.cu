// Implicit-GEMM convolution family on tcgen05 / TMEM / TMA for sm_100a, hand-written (no CUTLASS, no cuDNN):
//
//   FPROP   Y [pix, Cout]        = im2col(X)[pix, (r,s,ci)] . W[Cout, (r,s,ci)]^T          (+ fused BatchNorm statistics)
//   DGRAD   dX[pix, Cin]         = im2col(dY)[pix, (r,s,co)] . W[co, (R-1-r,S-1-s), Cin]    (stride 1)
//   WGRAD   dW[Cout, (r,s,ci)]  += dY[pix, Cout]^T . im2col(X)[pix, (r,s,ci)]               (fp32, split-K over pixels)
//
// Activations are NHWC bf16, filters are [Cout, R, S, Cin] bf16 (the channels-last bf16 shadow that the fused
// optimizer / aggregation kernels maintain), filter gradients accumulate in fp32 straight into the flat gradient
// buffer of the model.  1x1 / stride-1 layers and nn.Linear are the degenerate case (plain 2-D TMA tiles), so the same
// kernel is the dX = dY.W and dW = dY^T.X GEMM of the transformer layers.
//
// What makes it "implicit": the A operand of FPROP / DGRAD and the B operand of WGRAD are gathered by TMA **im2col**
// tensor maps (cuTensorMapEncodeIm2col): one `cp.async.bulk.tensor.4d...im2col` per (filter tap, 64-channel block)
// lands 128 (or 64) consecutive output pixels x 64 channels in shared memory, already SWIZZLE_128B, padding
// zero-filled and the convolution stride applied by the copy engine.  Nothing is ever unfolded in HBM.
//
// Operand layouts (UMMA shared-memory descriptors):
//   FPROP : A K-major (pixels x channels),  B K-major  (W rows = Cout, K contiguous)
//   DGRAD : A K-major,                      B MN-major (W[co][tap][ci]: ci = N contiguous, co = K rows)
//   WGRAD : A MN-major (dY[pix][co]: co = M contiguous, pix = K rows),  B MN-major (X[pix][ci])
// -> no transposed copy of the filter or of the activations exists anywhere.
//
// Structure (persistent, warp-specialised, 384 threads, one CTA per SM): warps 0-7 epilogue, warps 8 / 11 TMA producers
// (A / B operand), warp 9 MMA issuer, warp 10 TMEM allocator -- the single-thread pacing roles sit in the highest warp
// ids because the warp scheduler favours them there; smem ring of 192 KB, 2 TMEM accumulator stages.
// FPROP epilogue = bf16 tile through swizzled staging boxes + coalesced stores, and (optionally) the BatchNorm batch
// statistics of the layer: per-column sum / sum-of-squares of the bf16-rounded outputs, accumulated in registers over
// ALL row tiles of the CTA (a CTA keeps one column block), published once with fp64 reductions into L2; the last CTA
// of a column block to arrive does the per-channel finalize (mean, rstd, scale/bias, running statistics) from the
// totals.  The separate statistics pass over Y (bn.cu::bn_stats_kernel) disappears.
// WGRAD epilogue = the fp32 accumulators added into dW when a tile has one k-range; with several, every k-range stores its
// partial tile into its own workspace slice and wgrad_split_sum_kernel adds the slices into dW in one fixed order -- the
// same sum on every run (reductions in L2 would add them in arrival order).  Without it two runs of the same training
// drift apart within a few rounds and outputs of two builds cannot be compared.
#include <cuda.h>
#include <math.h>
#include <stdlib.h>
#include "common.cuh"
#include "api.h"

namespace igemm {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;
constexpr int UMMA_K = 16;
constexpr int kMaxStages = 8;
constexpr int kAccStages = 2;
constexpr int kTmemCols = 512;
constexpr int A_BYTES = BLOCK_M * BLOCK_K * 2;        // 16 KB
constexpr int RING_BYTES = 4 * (A_BYTES + 256 * 128); // 192 KB: 4 stages at N = 256, 6 at N = 128, 8 at N = 64
constexpr int BOX_BYTES = 64 * 128;                   // one 64-row x 64-element SWIZZLE_128B box (MN-major operands)
constexpr int kEpiWarps = 8;                          // 2 per TMEM lane quadrant: even / odd 32-column chunks
constexpr int STG_OFF = RING_BYTES;                   // epilogue staging: one 32 x 32 bf16 SWIZZLE_64B box (2 KB) x 2 per warp
constexpr int STG_BOX_BYTES = 32 * 64;
constexpr int STG_WARP_BYTES = 2 * STG_BOX_BYTES;
constexpr int BAR_OFF = STG_OFF + kEpiWarps * STG_WARP_BYTES;
constexpr int SMEM_BYTES = BAR_OFF + 1024 /*align slack*/ + 256 /*barriers*/;
static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB dynamic shared memory limit");
constexpr int kThreads = 128 + kEpiWarps * 32;
// Warp roles.  The warp scheduler of an SM sub-partition prefers the HIGHEST warp id among its eligible warps
// (B300_MICROARCH.md "Multi-warp arbiter"), so the single-thread roles that pace the main loop sit in the highest warps and
// the 8 epilogue warps below them: with the roles in warps 0-3 the busy epilogue starved the TMA / MMA threads and main
// loop and epilogue ran one after the other instead of overlapped (profiles/ncu_igemm_r2d.md).
constexpr int W_EPI0 = 0;        // warps 0..7: epilogue (TMEM lane quadrant = warp & 3)
constexpr int W_TMA_A = 8, W_MMA = 9, W_ALLOC = 10, W_TMA_B = 11;
constexpr int MAX_SLOTS = 148;

enum { FPROP = 0, DGRAD = 1, WGRAD = 2 };

struct Params {
    int M, N;                  // output space: FPROP/DGRAD [pixels, channels]; WGRAD [Cout, taps*Cin]
    int num_kb;                // 64-wide blocks of the whole reduction dimension
    int block_n;               // N tile (64/128/192/256); WGRAD: 256 (4 chunks of 64 columns)
    int a_im2col, b_im2col;    // operand gathered through an im2col tensor map (else plain tiled map)
    int PQ, Q;                 // output pixels per image / per image row of the im2col traversal
    int stride, pad;           // base pixel of output (p,q) = (p*stride - pad, q*stride - pad)
    int S;                     // filter width (tap = r*S + s)
    int cblocks;               // 64-channel blocks per filter tap
    int taps;                  // R*S
    int flip;                  // DGRAD: filter tap used = taps-1-tap
    int act;                   // bf16 epilogue: 0 none, 1 gelu(erf), 2 relu
    __nv_bfloat16* c_out;      // FPROP / DGRAD output [M, N] (row stride N)
    const float* bias;         // [N] or null
    const unsigned char* add_mask;  // [M, N/8] or null: 1 bit / element, add_src counts only where the bit is set (ReLU mask of the block output)
    const __nv_bfloat16* add_src;   // [M, N] or null: added to the result before the bf16 rounding (DGRAD: the gradient
                                    // that reaches the same tensor through the residual branch -> no separate add pass)
    // DGRAD of a stride-2 convolution: one work item = (output parity class, tile); a class (a, b) holds the dX pixels
    // (2i + a, 2j + b) and receives only the filter taps r = a + pad (mod 2), s = b + pad (mod 2): a stride-1 implicit
    // GEMM over dY with that sub-filter, rows scattered to the class' pixels by direct 64-byte stores.
    int dstride, ncls;
    int cls_ntap[4], cls_a[4], cls_b[4];
    unsigned char cls_off[4][4];     // dq | dp << 4 : im2col offset of the tap inside dY
    unsigned char cls_wtap[4][4];    // filter tap r * S + s
    int OH, OW, zero_fill;           // dX spatial size; zero_fill: also write zeros to the 3 pixels no tap reaches (1x1 / s2)
    __nv_bfloat16* dx;
    // WGRAD
    float* dw; long long ldw; int splits, kb_per_split; float out_scale;
    float* ws;                       // splits > 1: [splits][M][ldw] partial tiles, one slice per k-range
    // FPROP BatchNorm statistics (null gamma -> off)
    const float* gamma; const float* beta; float* running_mean; float* running_var; long long* num_batches_tracked;
    float* mean_out; float* rstd_out; float* scale_out; float* bias_out;
    float* part; int* counters; float eps, momentum;
    int stat_arrivals;       // CTAs that publish sums for one column block
};

V6_DEVINL float gelu_erf(float x) { return 0.5f * x * (1.f + erff(x * 0.70710678118654752f)); }

// Shared-memory operand descriptors, SWIZZLE_128B, split into a constant upper word and a lower word that carries the
// start address (so that the single MMA-issuing thread advances an operand with one 32-bit add):
//   K-major  (rows of 64 K-elements, 8-row groups 1024 B apart): SBO = 1024, LBO unused (1)
//   MN-major (64 MN-elements contiguous per K row, 8-row K groups 1024 B apart, 64-element MN chunks `lbo` apart)
// (MN-major form validated by glm_tc.cu, docs/ROUND2_PLAN.md appendix.)
constexpr uint32_t DESC_HI = (1024u >> 4) | (1u << 14) | (2u << 29);          // SBO | version 1 | SWIZZLE_128B
V6_DEVINL uint32_t desc_lo(uint32_t smem_addr, uint32_t lbo_bytes) { return ((smem_addr & 0x3FFFFu) >> 4) | ((lbo_bytes >> 4) << 16); }
V6_DEVINL uint64_t desc64(uint32_t lo) { return ((uint64_t)DESC_HI << 32) | lo; }
// D[tmem] (+)= A . B with both shared-memory descriptors assembled from their low words inside the asm block (no 64-bit
// shift / or in the issuing thread's instruction stream)
V6_DEVINL void umma_bf16_ss_lo(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tsetp.ne.b32 p, %4, 0;\n\tmov.b64 da, {%1, %5};\n\tmov.b64 db, {%2, %5};\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n\t}"
                 :: "r"(tmem_d), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(DESC_HI) : "memory");
}

V6_DEVINL void tma_load_im2col_4d(uint32_t smem_dst, const void* tmap, uint32_t bar, int c, int w, int h, int n, int off_w, int off_h) {
    const uint16_t ow = (uint16_t)off_w, oh = (uint16_t)off_h;
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.im2col.mbarrier::complete_tx::bytes"
                 " [%0], [%1, {%3, %4, %5, %6}], [%2], {%7, %8};"
                 :: "r"(smem_dst), "l"(tmap), "r"(bar), "r"(c), "r"(w), "r"(h), "r"(n), "h"(ow), "h"(oh) : "memory");
}
V6_DEVINL void tma_load_2d_u(uint32_t smem_dst, const void* tmap, uint32_t bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 :: "r"(smem_dst), "l"(tmap), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
V6_DEVINL void tma_load_3d_u(uint32_t smem_dst, const void* tmap, uint32_t bar, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 :: "r"(smem_dst), "l"(tmap), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
// explicit shared-state-space accesses for the epilogue's staging boxes (through generic pointers the compiler emitted
// LD.E / ST.E -- generic-address loads with global-memory-like latency, profiles/ncu_igemm_r2c.md)
V6_DEVINL void sts_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" :: "r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
V6_DEVINL uint4 lds_v4(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
    return v;
}
V6_DEVINL uint32_t lds_u32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
    return v;
}
V6_DEVINL float2 lds_f2(uint32_t addr) {
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr) : "memory");
    return v;
}
V6_DEVINL float lds_f1(uint32_t addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
    return v;
}
V6_DEVINL void sts_f2(uint32_t addr, float a, float b) { asm volatile("st.shared.v2.f32 [%0], {%1,%2};" :: "r"(addr), "f"(a), "f"(b) : "memory"); }
V6_DEVINL void epi_bar_sync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }      // the 8 epilogue warps only
V6_DEVINL void mbar_expect_tx_u(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
}
V6_DEVINL void umma_commit_u(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(bar) : "memory");
}
V6_DEVINL bool mbar_try_wait_u(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
V6_DEVINL void mbar_wait_u(uint32_t bar, uint32_t parity) {           // bounded: a deadlocked pipeline traps instead of hanging
    if (mbar_try_wait_u(bar, parity)) return;
    const long long t0 = clock64();
    uint32_t spins = 0;
    while (!mbar_try_wait_u(bar, parity)) {
        if ((++spins & 0xfff) == 0 && clock64() - t0 > 4000000000LL) { asm volatile("trap;"); }
    }
}

struct Item { int m_blk, n_blk, kb0, kb1, cls; };

// EPI (FPROP / DGRAD epilogue flavour, so that each instantiation carries only the code it runs -- the v2 kernel spent a
// fifth of its issue slots on instruction fetch and on branches around dead bias / GELU / scatter code):
//   EPI_PLAIN  bf16 tile -> staging -> TMA store
//   EPI_STATS  + BatchNorm statistics of the tile (FPROP)
//   EPI_GEN    bias / activation / add_src / stride-2 scatter
enum { EPI_PLAIN = 0, EPI_STATS = 1, EPI_GEN = 2 };

template <int MODE, int EPI>
__global__ void __launch_bounds__(kThreads, 1)
igemm_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
             const __grid_constant__ CUtensorMap tmap_c, const Params P) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);      // 1024-B aligned; derived by pointer arithmetic so that the compiler keeps the shared address space (LDS/STS, not generic LD/ST)
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + BAR_OFF);
    uint64_t* empty_bar = full_bar + kMaxStages;
    uint64_t* tfull_bar = empty_bar + kMaxStages;
    uint64_t* tempty_bar = tfull_bar + kAccStages;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + kAccStages);
    int* s_flag = reinterpret_cast<int*>(tmem_slot + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int num_m = (P.M + BLOCK_M - 1) / BLOCK_M;
    const int num_n = (P.N + P.block_n - 1) / P.block_n;
    const int num_tiles = num_m * num_n;
    const bool strided = MODE == DGRAD && P.dstride == 2;
    const int num_items = MODE == WGRAD ? num_tiles * P.splits : (strided ? num_tiles * P.ncls : num_tiles);
    // smem ring: a k-block = A tile (16 KB) + B tile (block_n rows of 128 B).  Narrow tiles put TWO k-blocks behind one
    // full / empty barrier pair: the single TMA thread and the single MMA thread pay their barrier round trips
    // (~100 cycles per try_wait / expect_tx / commit) per stage, and with 128 MMA cycles per k-block at N = 64 those round
    // trips -- not the tensor pipe, not L2 -- set the pace (profiles/ncu_igemm_r2b.md: 855 cycles per k-block).
    const int sub_bytes = A_BYTES + P.block_n * 128;
    const int ksub = (MODE != WGRAD && P.block_n <= 128) ? 2 : 1;
    const int stage_bytes = ksub * sub_bytes;
    const int num_stages = min(kMaxStages, RING_BYTES / stage_bytes);

    auto decode = [&](int item) {
        Item it;
        it.cls = 0;
        const int tile = (MODE == WGRAD || strided) ? item % num_tiles : item;
        if (EPI == EPI_STATS) {
            // n fastest and gridDim.x a multiple of num_n (host): a CTA stays on ONE column block for all of its row tiles, so
            // its per-channel running sums leave the registers once, at the end
            it.n_blk = tile % num_n;
            it.m_blk = tile / num_n;
        } else {
            it.m_blk = tile % num_m;                              // m fastest: concurrent CTAs share the filter block
            it.n_blk = tile / num_m;
        }
        if (MODE == WGRAD) {
            const int split = item / num_tiles;
            it.kb0 = split * P.kb_per_split;
            it.kb1 = min(P.num_kb, it.kb0 + P.kb_per_split);
        } else if (strided) {
            it.cls = item / num_tiles;                              // classes are ordered heaviest first by the host
            it.kb0 = 0; it.kb1 = P.cls_ntap[it.cls] * P.cblocks;
        } else { it.kb0 = 0; it.kb1 = P.num_kb; }
        return it;
    };
    // WGRAD: 64-column chunks of this N tile that exist (each chunk = one (tap, channel block))
    const int wch = P.block_n >> 6;                 // WGRAD: 64-column chunks per N tile (4, or 2 for block_n = 128)
    auto wgrad_chunks = [&](int n_blk) { return min(wch, (P.N >> 6) - n_blk * wch); };

    if (warp == W_TMA_A && lane == 0) { tma_prefetch_desc(&tmap_a); tma_prefetch_desc(&tmap_b); }
    if (warp == W_MMA && lane == 0) {
        for (int s = 0; s < kMaxStages; ++s) { mbar_init(&full_bar[s], 2); mbar_init(&empty_bar[s], 1); }      // full: A thread + B thread
        for (int s = 0; s < kAccStages; ++s) { mbar_init(&tfull_bar[s], 1); mbar_init(&tempty_bar[s], kEpiWarps); }
        mbar_fence_init();
    }
    if (warp == W_ALLOC) tmem_alloc<kTmemCols>(tmem_slot);
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // Programmatic dependent launch: everything above (barrier init, TMEM allocation, descriptor prefetch) overlaps the
    // tail of the previous kernel in the stream; from here on this grid reads what that kernel wrote.  Dependents are
    // released right away -- they park in their own griddepcontrol.wait until this grid has completed and flushed.
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const uint32_t smem0 = smem_u32(smem);
    const uint32_t full0 = smem_u32(full_bar), empty0 = smem_u32(empty_bar);

    if (warp == W_TMA_A || warp == W_TMA_B) {
        // ============================ TMA producers ============================
        // Two threads: warp 0 loads the A operand of every stage, warp 3 the B operand; each arms the stage's full barrier
        // with its own byte count.  (One thread issuing all copies of a k-block -- up to 6 for WGRAD -- was the pace
        // setter of the narrow-tile and WGRAD main loops.)
        if (lane == 0) {
            const bool is_a = warp == W_TMA_A;
            int stage = 0; uint32_t phase = 0;
            for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
                const Item it = decode(item);
                const int m0 = it.m_blk * BLOCK_M;
                if (MODE != WGRAD) {
                    int pn = 0, pw = 0, ph = 0;                  // base pixel of the tile's first row (im2col A operand)
                    if (P.a_im2col) {
                        pn = m0 / P.PQ;
                        const int rem = m0 - pn * P.PQ;
                        ph = (rem / P.Q) * P.stride - P.pad;
                        pw = (rem % P.Q) * P.stride - P.pad;
                    }
                    const int n0 = it.n_blk * P.block_n;
                    const int nch = P.block_n >> 6;
                    const uint32_t tx = is_a ? A_BYTES : (MODE == FPROP ? P.block_n * 128 : nch * BOX_BYTES);
                    int tap = 0, tap_s = 0, tap_r = 0, cb = 0;   // k-block = (filter tap, 64-channel block), advanced incrementally
                    if (strided) { tap_s = P.cls_off[it.cls][0] & 15; tap_r = P.cls_off[it.cls][0] >> 4; }
                    for (int kb = 0; kb < it.kb1; kb += ksub) {
                        const uint32_t fb = full0 + stage * 8;
                        const int nsub = min(ksub, it.kb1 - kb);
                        mbar_wait_u(empty0 + stage * 8, phase ^ 1);
                        mbar_expect_tx_u(fb, nsub * tx);
                        for (int u = 0; u < nsub; ++u) {
                            const uint32_t sa = smem0 + stage * stage_bytes + u * sub_bytes, sb = sa + A_BYTES;
                            if (is_a) {
                                if (P.a_im2col) tma_load_im2col_4d(sa, &tmap_a, fb, cb * 64, pw, ph, pn, tap_s, tap_r);
                                else tma_load_2d_u(sa, &tmap_a, fb, (kb + u) * BLOCK_K, m0);
                            } else if (MODE == FPROP) {
                                tma_load_2d_u(sb, &tmap_b, fb, (kb + u) * BLOCK_K, n0);
                            } else {
                                const int wtap = strided ? P.cls_wtap[it.cls][tap] : (P.flip ? P.taps - 1 - tap : tap);
                                for (int j = 0; j < nch; ++j) tma_load_3d_u(sb + j * BOX_BYTES, &tmap_b, fb, n0 + j * 64, wtap, cb * 64);
                            }
                            if (++cb == P.cblocks) {
                                cb = 0; ++tap;
                                if (strided) { const int o = P.cls_off[it.cls][tap & 3]; tap_s = o & 15; tap_r = o >> 4; }
                                else if (++tap_s == P.S) { tap_s = 0; ++tap_r; }
                            }
                        }
                        if (++stage == num_stages) { stage = 0; phase ^= 1; }
                    }
                } else {
                    const int na = min(2, (P.M - m0 + 63) >> 6);
                    const int nch = wgrad_chunks(it.n_blk);
                    int cs[4], cr[4], cc[4];                     // (tap_s, tap_r, channel block) of the tile's column chunks
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int chunk = it.n_blk * wch + j, tap = chunk / P.cblocks;
                        cc[j] = (chunk - tap * P.cblocks) * 64; cs[j] = tap % P.S; cr[j] = tap / P.S;
                    }
                    const uint32_t tx = (is_a ? na : nch) * BOX_BYTES;
                    for (int kb = it.kb0; kb < it.kb1; ++kb) {
                        const uint32_t fb = full0 + stage * 8;
                        mbar_wait_u(empty0 + stage * 8, phase ^ 1);
                        const uint32_t sa = smem0 + stage * stage_bytes, sb = sa + A_BYTES;
                        mbar_expect_tx_u(fb, tx);
                        const int pix0 = kb * BLOCK_K;
                        if (is_a) {
                            for (int i = 0; i < na; ++i) tma_load_2d_u(sa + i * BOX_BYTES, &tmap_a, fb, m0 + i * 64, pix0);
                        } else if (P.b_im2col) {
                            const int bn = pix0 / P.PQ, rem = pix0 - bn * P.PQ;
                            const int bh = (rem / P.Q) * P.stride - P.pad, bw = (rem % P.Q) * P.stride - P.pad;
#pragma unroll
                            for (int j = 0; j < 4; ++j)
                                if (j < nch) tma_load_im2col_4d(sb + j * BOX_BYTES, &tmap_b, fb, cc[j], bw, bh, bn, cs[j], cr[j]);
                        } else {
#pragma unroll
                            for (int j = 0; j < 4; ++j)
                                if (j < nch) tma_load_2d_u(sb + j * BOX_BYTES, &tmap_b, fb, (it.n_blk * wch + j) * 64, pix0);
                        }
                        if (++stage == num_stages) { stage = 0; phase ^= 1; }
                    }
                }
            }
        }
    } else if (warp == W_MMA) {
        // ============================ MMA issuer (one thread) ==============================
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            const uint32_t tfull0 = smem_u32(tfull_bar), tempty0 = smem_u32(tempty_bar);
            // per-k-step advance of the descriptor start address (>> 4): K-major 16 elements = 32 B; MN-major 16 K rows = 2048 B
            constexpr uint32_t a_step = MODE == WGRAD ? (2048u >> 4) : (32u >> 4);
            constexpr uint32_t b_step = MODE == FPROP ? (32u >> 4) : (2048u >> 4);
            const uint32_t a_lo0 = desc_lo(smem0, MODE == WGRAD ? BOX_BYTES : 16), b_lo0 = desc_lo(smem0 + A_BYTES, MODE == FPROP ? 16 : BOX_BYTES);
            const uint32_t stage_step = (uint32_t)stage_bytes >> 4;
            for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
                const Item it = decode(item);
                const int n_umma = MODE == WGRAD ? wgrad_chunks(it.n_blk) * 64 : P.block_n;
                uint32_t idesc = make_idesc_bf16(BLOCK_M, n_umma);
                if (MODE == DGRAD) idesc |= 1u << 16;                       // B MN-major
                if (MODE == WGRAD) idesc |= (1u << 15) | (1u << 16);        // A and B MN-major
                mbar_wait_u(tempty0 + acc * 8, acc_phase ^ 1);
                tcgen05_fence_after();
                const uint32_t d_tmem = tmem_base + acc * 256;
                uint32_t accumulate = 0;
                const uint32_t sub_step = (uint32_t)sub_bytes >> 4;
                for (int kb = it.kb0; kb < it.kb1; kb += ksub) {
                    const int nsub = min(ksub, it.kb1 - kb);
                    mbar_wait_u(full0 + stage * 8, phase);
                    tcgen05_fence_after();
                    uint32_t a_lo = a_lo0 + stage * stage_step, b_lo = b_lo0 + stage * stage_step;
                    for (int u = 0; u < nsub; ++u) {
#pragma unroll
                        for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
                            umma_bf16_ss_lo(d_tmem, a_lo + k * a_step, b_lo + k * b_step, idesc, accumulate);
                            accumulate = 1;
                        }
                        a_lo += sub_step; b_lo += sub_step;
                    }
                    umma_commit_u(empty0 + stage * 8);
                    if (kb + nsub >= it.kb1) umma_commit_u(tfull0 + acc * 8);
                    if (++stage == num_stages) { stage = 0; phase ^= 1; }
                }
                if (++acc == kAccStages) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else if (warp < kEpiWarps) {
        // ============================ epilogue (8 warps) ================================
        const int quad = warp & 3;                    // TMEM lanes [32*quad, 32*quad+32)
        const int half = warp >> 2;             // this warp takes the 32-column chunks with (chunk & 1) == half
        const int et = warp * 32 + lane;        // epilogue thread id 0..255: owns column `et` of the statistics
        constexpr bool stats = MODE == FPROP && EPI == EPI_STATS;
        int acc = 0; uint32_t acc_phase = 0;
        float run1[4][2], run2[4][2];                 // running column sums of this warp's (<= 4) chunks: lanes 0..15 own a column pair
#pragma unroll
        for (int k = 0; k < 4; ++k) run1[k][0] = run1[k][1] = run2[k][0] = run2[k][1] = 0.f;
        const uint32_t stg = smem0 + STG_OFF + warp * STG_WARP_BYTES;      // shared-space address of this warp's two boxes
        const int nck = P.block_n >> 6;               // 32-column chunks of a tile this warp handles (chunk index 2k + half)

        // fp32 accumulator row (32 columns) -> packed bf16 (EPI_GEN: + bias / residual-gradient add / activation)
        auto finish = [&](const uint32_t (&v)[32], uint32_t (&packed)[16], int row, int col0) {
            if (EPI != EPI_GEN) {
#pragma unroll
                for (int j = 0; j < 16; ++j) packed[j] = pack_bf16x2(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
                return;
            }
            float f[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
            if (P.bias) {
#pragma unroll
                for (int j = 0; j < 32; ++j) if (col0 + j < P.N) f[j] += __ldg(P.bias + col0 + j);
            }
            if (P.act == 1) {
#pragma unroll
                for (int j = 0; j < 32; ++j) f[j] = gelu_erf(f[j]);
            } else if (P.act == 2) {
#pragma unroll
                for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j], 0.f);
            }
#pragma unroll
            for (int j = 0; j < 16; ++j) packed[j] = pack_bf16x2(f[2 * j], f[2 * j + 1]);
        };
        // [32 rows][32 bf16 = 64 B] staging box, SWIZZLE_64B: 16-byte chunk j of row r sits at chunk j ^ ((r >> 1) & 3)
        auto to_box = [&](uint32_t sbox, const uint32_t (&packed)[16]) {
            const uint32_t rowa = sbox + lane * 64, sw = (lane >> 1) & 3;
#pragma unroll
            for (int j = 0; j < 4; ++j)
                sts_v4(rowa + ((j ^ sw) << 4), packed[4 * j], packed[4 * j + 1], packed[4 * j + 2], packed[4 * j + 3]);
        };
        // staging box -> global memory: 4 lanes cover one row's 64 bytes (two full 32-byte sectors), 8 rows per instruction.
        // (v2 used a TMA store per box: its proxy fence + store-read wait sat on the critical path of every chunk and the
        // short-K layers are bound by exactly this chain -- profiles/ncu_igemm_r2b.md.)
        auto box_to_global = [&](uint32_t sbox, int row0, int c0) {
            const int ch = lane & 3;
            if (c0 + ch * 8 >= P.N) return;
            const size_t off = (size_t)(row0 + (lane >> 2)) * P.N + c0 + ch * 8;
            uint4 val[4], addv[4];
            const bool add = EPI == EPI_GEN && P.add_src != nullptr;
            unsigned mbits[4] = {0xffu, 0xffu, 0xffu, 0xffu};
            if (add) {      // the gradient of the residual branch, read with the same fully coalesced pattern as the store
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const bool in = row0 + (lane >> 2) + 8 * i < P.M;
                    addv[i] = in ? __ldg(reinterpret_cast<const uint4*>(P.add_src + off + (size_t)(8 * i) * P.N)) : make_uint4(0u, 0u, 0u, 0u);
                    // the branch gradient is dy . relu'(block output): the mask byte of these 8 channels instead of a masked copy
                    if (P.add_mask && in) mbits[i] = __ldg(P.add_mask + (off + (size_t)(8 * i) * P.N) / 8);
                }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int r = (lane >> 2) + 8 * i;
                val[i] = lds_v4(sbox + r * 64 + ((ch ^ ((r >> 1) & 3)) << 4));
            }
            if (add) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    uint32_t* v = reinterpret_cast<uint32_t*>(&val[i]);
                    const uint32_t* q = reinterpret_cast<const uint32_t*>(&addv[i]);
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const float2 x = unpack_bf16x2(v[e]), y = unpack_bf16x2(q[e]);
                        v[e] = pack_bf16x2(x.x + (((mbits[i] >> (2 * e)) & 1u) ? y.x : 0.f), x.y + (((mbits[i] >> (2 * e + 1)) & 1u) ? y.y : 0.f));
                    }
                }
            }
            __nv_bfloat16* dst = P.c_out + off;
#pragma unroll
            for (int i = 0; i < 4; ++i)
                if (row0 + (lane >> 2) + 8 * i < P.M) *reinterpret_cast<uint4*>(dst + (size_t)(8 * i) * P.N) = val[i];
        };
        // column sums of the bf16-rounded box: lanes 0..15 take rows 0..15, lanes 16..31 rows 16..31 of column pair
        // (lane & 15); the halves meet through one shuffle; added to the running sums of chunk slot k
        auto box_stats = [&](uint32_t sbox, int k) {
            const int cp = lane & 15, r0 = (lane >> 4) * 16;
            float a0 = 0.f, a1 = 0.f, b0 = 0.f, b1 = 0.f;
            const uint32_t base = sbox + r0 * 64 + (cp & 3) * 4;
#pragma unroll
            for (int r = 0; r < 16; ++r) {
                // row r0 + r: r0 is a multiple of 16, so the swizzle term only depends on r
                const uint32_t wv = lds_u32(base + r * 64 + ((((uint32_t)cp >> 2) ^ ((r >> 1) & 3)) << 4));
                const float x0 = __uint_as_float(wv << 16), x1 = __uint_as_float(wv & 0xffff0000u);
                a0 += x0; a1 += x1; b0 = fmaf(x0, x0, b0); b1 = fmaf(x1, x1, b1);
            }
            a0 += __shfl_xor_sync(0xffffffffu, a0, 16); a1 += __shfl_xor_sync(0xffffffffu, a1, 16);
            b0 += __shfl_xor_sync(0xffffffffu, b0, 16); b1 += __shfl_xor_sync(0xffffffffu, b1, 16);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk)
                if (kk == k) { run1[kk][0] += a0; run1[kk][1] += a1; run2[kk][0] += b0; run2[kk][1] += b1; }
        };
        // stride-2 DGRAD: row (n, i, j) of the class grid -> dX pixel (2i + a, 2j + b).  Through the staging box like the
        // dense path: 4 lanes cover the 64 bytes of one pixel's 32 channels (two full sectors), 8 pixels per instruction
        // (one thread per pixel writing 4 x 16 B at a 2-pixel pitch was 4x the LSU transactions); the pixels of the
        // classes no tap reaches (1x1 filters) are zero-filled with the same pattern.
        auto box_scatter = [&](uint32_t sbox, int row0, int c0, int cls) {
            const int ch = lane & 3;
            if (c0 + ch * 8 >= P.N) return;
            __nv_bfloat16* base = P.dx + c0 + ch * 8;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int r = (lane >> 2) + 8 * i, m = row0 + r;
                if (m >= P.M) continue;
                const uint4 val = lds_v4(sbox + r * 64 + ((ch ^ ((r >> 1) & 3)) << 4));
                const int n_img = m / P.PQ, rem = m - n_img * P.PQ;
                const int qi = rem / P.Q, oi = 2 * qi, oj = 2 * (rem - qi * P.Q);
                __nv_bfloat16* img = base + ((size_t)n_img * P.OH * P.OW) * P.N;
                *reinterpret_cast<uint4*>(img + ((size_t)(oi + P.cls_a[cls]) * P.OW + oj + P.cls_b[cls]) * P.N) = val;
                if (P.zero_fill) {
#pragma unroll
                    for (int z = 1; z < 4; ++z)
                        *reinterpret_cast<uint4*>(img + ((size_t)(oi + (z >> 1)) * P.OW + oj + (z & 1)) * P.N) = make_uint4(0u, 0u, 0u, 0u);
                }
            }
        };

        for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
            const Item it = decode(item);
            mbar_wait(&tfull_bar[acc], acc_phase);
            tcgen05_fence_after();
            const uint32_t t_row = tmem_base + acc * 256 + ((uint32_t)(quad * 32) << 16);
            if (MODE == WGRAD) {
                // fp32 accumulators -> dW[row][n_blk*block_n + col] (+=); row = output channel.  With ONE k-range per tile the
                // tile owns its output and a plain load-add-store does it; with several, this k-range's partial tile goes to its
                // workspace slice with plain stores (wgrad_split_sum_kernel adds the slices in a fixed order) -- no L2 reductions, which
                // run at ~0.7 TB/s, an order of magnitude below plain stores (profiles/kernel_bench_linear_bwd_r2.txt)
                const int row = it.m_blk * BLOCK_M + quad * 32 + lane;
                const int ncols = wgrad_chunks(it.n_blk) * 64;
                const bool owned = P.splits == 1;
                float* drow = (owned ? P.dw : P.ws + (long long)(it.kb0 / P.kb_per_split) * P.M * P.ldw)
                              + (long long)row * P.ldw + it.n_blk * P.block_n;
#pragma unroll 1
                for (int c = half * 32; c < ncols; c += 64) {
                    uint32_t v[32];
                    tmem_ld_32x32b_x32(t_row + c, v);
                    tmem_ld_wait();
                    if (row < P.M) {
                        if (owned) {
                            float4 o[8];
#pragma unroll
                            for (int j = 0; j < 8; ++j) o[j] = *reinterpret_cast<const float4*>(drow + c + 4 * j);
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                o[j].x = fmaf(__uint_as_float(v[4 * j]), P.out_scale, o[j].x); o[j].y = fmaf(__uint_as_float(v[4 * j + 1]), P.out_scale, o[j].y);
                                o[j].z = fmaf(__uint_as_float(v[4 * j + 2]), P.out_scale, o[j].z); o[j].w = fmaf(__uint_as_float(v[4 * j + 3]), P.out_scale, o[j].w);
                                *reinterpret_cast<float4*>(drow + c + 4 * j) = o[j];
                            }
                        } else {
#pragma unroll
                            for (int j = 0; j < 32; j += 4)
                                *reinterpret_cast<float4*>(drow + c + j) = make_float4(
                                    __uint_as_float(v[j]) * P.out_scale, __uint_as_float(v[j + 1]) * P.out_scale,
                                    __uint_as_float(v[j + 2]) * P.out_scale, __uint_as_float(v[j + 3]) * P.out_scale);
                        }
                    }
                }
            } else {
                const int row0 = it.m_blk * BLOCK_M + quad * 32;
                const int colb = it.n_blk * P.block_n + half * 32;          // first column of this warp's chunk 0
                const bool rows_ok = row0 < P.M;
                int k = 0;
                // two chunks per iteration: both TMEM loads, conversions, box writes and TMA stores in flight together
#pragma unroll 1
                for (; k + 1 < nck; k += 2) {
                    uint32_t v0[32], v1[32];
                    tmem_ld_32x32b_x32(t_row + half * 32 + k * 64, v0);
                    tmem_ld_32x32b_x32(t_row + half * 32 + k * 64 + 64, v1);
                    tmem_ld_wait();
                    const int c0 = colb + k * 64, c1 = c0 + 64;
                    if (!rows_ok || c0 >= P.N) continue;                     // warp-uniform
                    const bool second = c1 < P.N;
                    uint32_t p0[16], p1[16];
                    finish(v0, p0, row0 + lane, c0);
                    finish(v1, p1, row0 + lane, c1);
                    __syncwarp();                                            // every lane is done reading the boxes of the previous pair
                    to_box(stg, p0);
                    to_box(stg + STG_BOX_BYTES, p1);
                    __syncwarp();
                    if (EPI == EPI_GEN && strided) {
                        box_scatter(stg, row0, c0, it.cls);
                        if (second) box_scatter(stg + STG_BOX_BYTES, row0, c1, it.cls);
                        continue;
                    }
                    box_to_global(stg, row0, c0);
                    if (second) box_to_global(stg + STG_BOX_BYTES, row0, c1);
                    if (stats) { box_stats(stg, k); if (second) box_stats(stg + STG_BOX_BYTES, k + 1); }
                }
                if (k < nck) {                                               // odd chunk count (block_n = 64 / 192)
                    uint32_t v0[32];
                    tmem_ld_32x32b_x32(t_row + half * 32 + k * 64, v0);
                    tmem_ld_wait();
                    const int c0 = colb + k * 64;
                    if (rows_ok && c0 < P.N) {
                        uint32_t p0[16];
                        finish(v0, p0, row0 + lane, c0);
                        __syncwarp();
                        to_box(stg, p0);
                        __syncwarp();
                        if (EPI == EPI_GEN && strided) {
                            box_scatter(stg, row0, c0, it.cls);
                        } else {
                            box_to_global(stg, row0, c0);
                            if (stats) box_stats(stg, k);
                        }
                    }
                }
            }
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty_bar[acc]);
            if (++acc == kAccStages) { acc = 0; acc_phase ^= 1; }

            if (stats) {
                const int nxt = item + gridDim.x;
                const bool flush = nxt >= num_items || decode(nxt).n_blk != it.n_blk;
                if (flush) {
                    // combine the 8 warps' running sums through the (now idle) staging boxes and add this CTA's totals to the
                    // column block's; the last CTA to arrive finalizes
                    __syncwarp();
                    // this warp's box area doubles as scratch: [chunk k][sum | sumsq][32 columns] floats = 1 KB of the 4 KB
                    if (lane < 16) {
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            sts_f2(stg + (k * 64 + 2 * lane) * 4, run1[k][0], run1[k][1]);
                            sts_f2(stg + (k * 64 + 32 + 2 * lane) * 4, run2[k][0], run2[k][1]);
                        }
                    }
#pragma unroll
                    for (int k = 0; k < 4; ++k) run1[k][0] = run1[k][1] = run2[k][0] = run2[k][1] = 0.f;
                    epi_bar_sync();
                    double* sums = reinterpret_cast<double*>(P.part) + (size_t)it.n_blk * P.block_n * 2;
                    if (et < P.block_n) {
                        const int ch = et >> 5, hh = ch & 1, kk = ch >> 1, ci = et & 31;
                        float t1 = 0.f, t2 = 0.f;
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const uint32_t ws = smem0 + STG_OFF + (hh * 4 + q) * STG_WARP_BYTES;
                            t1 += lds_f1(ws + (kk * 64 + ci) * 4); t2 += lds_f1(ws + (kk * 64 + 32 + ci) * 4);
                        }
                        // this CTA's sums of its whole run of row tiles meet the other CTAs' in L2 (fp64 reductions: the
                        // arrival order only moves the 16th digit); nothing is folded serially by anybody
                        asm volatile("red.global.add.f64 [%0], %1;" :: "l"(sums + et), "d"((double)t1) : "memory");
                        asm volatile("red.global.add.f64 [%0], %1;" :: "l"(sums + P.block_n + et), "d"((double)t2) : "memory");
                    }
                    __threadfence();
                    epi_bar_sync();                                       // sums published; staging boxes free again
                    if (et == 0) {
                        int old;
                        asm volatile("atom.add.acq_rel.gpu.global.s32 %0, [%1], 1;" : "=r"(old) : "l"(P.counters + it.n_blk) : "memory");
                        const int last = old == P.stat_arrivals - 1;
                        if (last) P.counters[it.n_blk] = 0;              // every expected arrival has happened
                        *s_flag = last;
                    }
                    epi_bar_sync();
                    const bool last = *s_flag != 0;
                    epi_bar_sync();                                      // s_flag may be rewritten by the next flush
                    if (last && et < P.block_n) {
                        const double t1 = __ldcg(sums + et), t2 = __ldcg(sums + P.block_n + et);
                        __stcg(sums + et, 0.0);                          // self-resetting, like the counters
                        __stcg(sums + P.block_n + et, 0.0);
                        const int c = it.n_blk * P.block_n + et;
                        if (c < P.N) {
                            const double invR = 1.0 / (double)P.M;
                            const double mean_d = t1 * invR;
                            double var_d = t2 * invR - mean_d * mean_d;
                            if (var_d < 0.0) var_d = 0.0;
                            const float mean = (float)mean_d, var = (float)var_d;
                            const float rstd = rsqrtf(var + P.eps);
                            P.mean_out[c] = mean;
                            P.rstd_out[c] = rstd;
                            const float sc = P.gamma[c] * rstd;
                            P.scale_out[c] = sc;
                            P.bias_out[c] = P.beta[c] - mean * sc;
                            if (P.running_mean) {
                                const float unbiased = P.M > 1 ? var * (float)P.M / (float)(P.M - 1) : var;
                                P.running_mean[c] = (1.f - P.momentum) * P.running_mean[c] + P.momentum * mean;
                                P.running_var[c] = (1.f - P.momentum) * P.running_var[c] + P.momentum * unbiased;
                            }
                            if (P.num_batches_tracked && c == 0) *P.num_batches_tracked += 1;
                        }
                    }
                }
            }
        }
    }

    tcgen05_fence_before();
    __syncthreads();
    if (warp == W_ALLOC) { tcgen05_fence_after(); tmem_dealloc<kTmemCols>(tmem_base); }
}

}  // namespace igemm

// ------------------------------------------------------------------------------------------------- host side
extern "C" long long v6_igemm_scratch_floats() { return 64 + (long long)2048 * 2 * 2; }   // counters | fp64 [sum | sumsq] per channel

namespace {

struct ConvGeom {
    int N, H, W, C;          // the im2col-side activation tensor (NHWC)
    int R, S, stride, pad;   // filter window / traversal over that tensor
    int P, Q;                // traversal output size
    long long pitch_w = 0, pitch_h = 0, pitch_n = 0;      // byte pitches (0 = dense)
};

typedef void (*KernelFn)(const CUtensorMap, const CUtensorMap, const CUtensorMap, const igemm::Params);

// one instantiation per (mode, epilogue flavour) that is actually used
KernelFn pick_kernel(int mode, int epi) {
    using namespace igemm;
    if (mode == FPROP) return epi == EPI_STATS ? igemm_kernel<FPROP, EPI_STATS> : epi == EPI_GEN ? igemm_kernel<FPROP, EPI_GEN> : igemm_kernel<FPROP, EPI_PLAIN>;
    if (mode == DGRAD) return epi == EPI_GEN ? igemm_kernel<DGRAD, EPI_GEN> : igemm_kernel<DGRAD, EPI_PLAIN>;
    return igemm_kernel<WGRAD, EPI_PLAIN>;
}

int set_smem_attr() {
    static bool done = false;
    if (!done) {
        using namespace igemm;
        const int combos[6][2] = {{FPROP, EPI_PLAIN}, {FPROP, EPI_STATS}, {FPROP, EPI_GEN}, {DGRAD, EPI_PLAIN}, {DGRAD, EPI_GEN}, {WGRAD, EPI_PLAIN}};
        for (auto& c : combos) {
            cudaError_t e = cudaFuncSetAttribute(pick_kernel(c[0], c[1]), cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
            if (e != cudaSuccess) return (int)e;
        }
        done = true;
    }
    return 0;
}

int im2col_map(void* out, const void* ptr, const ConvGeom& g, int pixels) {
    return v6_make_tmap_im2col_bf16(out, (uint64_t)ptr, g.C, g.W, g.H, g.N, -g.pad, -g.pad, g.pad - (g.S - 1), g.pad - (g.R - 1), 64, pixels,
                                    g.stride, g.stride, (uint64_t)g.pitch_w, (uint64_t)g.pitch_h, (uint64_t)g.pitch_n);
}

// N-tile width from a small cost model (cycles, fitted to profiles/conv_probe_time_r2b.jsonl): a tile's main loop costs
// num_kb x max(MMA issue time, operand fetch time) and its epilogue (BN / 64) store chains per warp; the two overlap
// (2 TMEM accumulator stages), tiles run in waves of one per SM.
int pick_block_n(int M, int N, int num_kb = 8, bool stats = false) {
    const long long num_m = (M + 127) / 128;
    if (N <= 64) return 64;
    int best = 64;
    double best_t = 1e30;
    for (int bn : {256, 128, 64}) {
        if (bn > 64 && N < bn && N % bn != 0 && N <= bn / 2) continue;
        const long long tiles = num_m * ((N + bn - 1) / bn);
        const double waves = (double)((tiles + 147) / 148);
        const double mma = 2.0 * bn, fetch = (16384.0 + bn * 128.0) / 60.0;
        const double main_loop = num_kb * (mma > fetch ? mma : fetch) + 600.0;
        const double epi = (bn / 64) * (stats ? 1500.0 : 900.0) * 0.5 + 300.0;      // pairs of chunks per chain
        const double t = waves * (main_loop > epi ? main_loop : epi);
        if (t < best_t * 0.97) { best_t = t; best = bn; }
    }
    return best;
}

int launch(int mode, const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const igemm::Params& P, cudaStream_t s) {
    using namespace igemm;
    int rc = set_smem_attr();
    if (rc) return rc;
    const int num_m = (P.M + BLOCK_M - 1) / BLOCK_M, num_n = (P.N + P.block_n - 1) / P.block_n;
    const int items = mode == WGRAD ? num_m * num_n * P.splits : (mode == DGRAD && P.dstride == 2 ? num_m * num_n * P.ncls : num_m * num_n);
    static int sms = 0;
    if (!sms) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev); if (sms <= 0) sms = 148; }
    const int cap = sms < MAX_SLOTS ? sms : MAX_SLOTS;
    int grid = items < cap ? items : cap;
    int epi = EPI_PLAIN;
    if (mode == FPROP) epi = P.gamma ? EPI_STATS : ((P.bias || P.act) ? EPI_GEN : EPI_PLAIN);
    else if (mode == DGRAD) epi = (P.dstride == 2 || P.add_src) ? EPI_GEN : EPI_PLAIN;
    igemm::Params Pl = P;
    if (epi == EPI_STATS) {      // every CTA keeps one column block (see decode): grid = whole groups of num_n CTAs
        grid = items < cap ? items : (cap / num_n) * num_n;
        Pl.stat_arrivals = grid / num_n;
    }
    static const bool pdl = [] { const char* e = getenv("V6B200_PDL"); return !(e && e[0] == '0'); }();
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = SMEM_BYTES;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    cudaError_t le = cudaLaunchKernelEx(&cfg, pick_kernel(mode, epi), ta, tb, tc, Pl);
    if (le != cudaSuccess) return (int)le;
    V6_CHECK_LAUNCH();
    return 0;
}

}  // namespace

// y[N,P,Q,Cout] = conv(x[N,H,W,Cin], w[Cout,R,S,Cin]); bn != 0: also the BatchNorm batch statistics of y (see Params)
extern "C" int v6_conv_fprop(const void* x, const void* w, void* y, const float* bias, int act, int N, int H, int W, int Cin, int Cout,
                             int R, int S, int stride, int pad, const float* gamma, const float* beta, float* running_mean,
                             float* running_var, long long* num_batches_tracked, float* mean_out, float* rstd_out,
                             float* scale_bias_out, float* scratch, float eps, float momentum, int force_im2col, long long pitch_w,
                             long long pitch_h, long long pitch_n, cudaStream_t stream) {
    using namespace igemm;
    if (Cin % 64 != 0 || Cout % 8 != 0 || (R != S && pad != 0)) return (int)cudaErrorInvalidValue;
    const int Pp = (H + 2 * pad - R) / stride + 1, Qq = (W + 2 * pad - S) / stride + 1;
    const long long Mll = (long long)N * Pp * Qq;
    if (Mll >= (1LL << 31)) return (int)cudaErrorInvalidValue;
    const int M = (int)Mll, K = R * S * Cin;
    const bool plain = R == 1 && S == 1 && stride == 1 && pad == 0 && !force_im2col && !pitch_w;
    Params P = {};
    P.M = M; P.N = Cout; P.num_kb = K / 64; P.block_n = pick_block_n(M, Cout, K / 64, gamma != nullptr);
    P.a_im2col = plain ? 0 : 1; P.PQ = Pp * Qq; P.Q = Qq; P.stride = stride; P.pad = pad; P.S = S; P.cblocks = Cin / 64; P.taps = R * S;
    P.act = act; P.bias = bias; P.c_out = (__nv_bfloat16*)y;
    if (gamma) {
        if (Cout % 64 != 0) return (int)cudaErrorInvalidValue;
        P.gamma = gamma; P.beta = beta; P.running_mean = running_mean; P.running_var = running_var;
        P.num_batches_tracked = num_batches_tracked; P.mean_out = mean_out; P.rstd_out = rstd_out;
        P.scale_out = scale_bias_out; P.bias_out = scale_bias_out + Cout; P.eps = eps; P.momentum = momentum;
        P.counters = reinterpret_cast<int*>(scratch); P.part = scratch + 64;
        const int num_n = (Cout + P.block_n - 1) / P.block_n;
        if (num_n > 64 || (long long)num_n * P.block_n > 2048) return (int)cudaErrorInvalidValue;
    }
    alignas(64) CUtensorMap ta, tb, tc;
    if (plain) { if (v6_make_tmap_2d_bf16(&ta, (uint64_t)x, M, Cin, (uint64_t)Cin * 2, BLOCK_M, BLOCK_K, 1)) return -2; }
    else { ConvGeom g{N, H, W, Cin, R, S, stride, pad, Pp, Qq, pitch_w, pitch_h, pitch_n}; if (im2col_map(&ta, x, g, BLOCK_M)) return -2; }
    if (v6_make_tmap_2d_bf16(&tb, (uint64_t)w, Cout, K, (uint64_t)K * 2, P.block_n, BLOCK_K, 1)) return -2;
    if (v6_make_tmap_2d_bf16(&tc, (uint64_t)y, M, Cout, (uint64_t)Cout * 2, 32, 32, 2)) return -2;      // 32 x 32 boxes, SWIZZLE_64B
    return launch(FPROP, ta, tb, tc, P, stream);
}

// dx[N,H,W,Cin] = conv_transpose(dy[N,P,Q,Cout], w[Cout,R,S,Cin]) for stride 1 (P = H + 2*pad - R + 1)
extern "C" int v6_conv_dgrad(const void* dy, const void* w, void* dx, int N, int H, int W, int Cin, int Cout, int R, int S, int stride,
                             int pad, int force_im2col, const void* add_src, const void* add_mask, cudaStream_t stream) {
    using namespace igemm;
    if (Cout % 64 != 0 || Cin % 8 != 0 || R != S) return (int)cudaErrorInvalidValue;
    if (add_src && (stride != 1 || Cin % 32 != 0)) return (int)cudaErrorInvalidValue;
    alignas(64) CUtensorMap ta, tb, tc;
    {
        const uint64_t dims[3] = {(uint64_t)Cin, (uint64_t)(R * S), (uint64_t)Cout};
        const uint64_t strides[2] = {(uint64_t)Cin * 2, (uint64_t)R * S * Cin * 2};
        const uint32_t box[3] = {64, 1, 64};
        if (v6_make_tmap_tiled_bf16(&tb, (uint64_t)w, 3, dims, strides, box, 1)) return -2;
    }
    Params P = {};
    if (stride == 2) {
        // 3x3 / pad 1 (4 parity classes with 1, 2, 2, 4 taps) and 1x1 / pad 0 (one class, the other pixels are zeros)
        if (!((R == 3 && pad == 1) || (R == 1 && pad == 0)) || (H & 1) || (W & 1)) return (int)cudaErrorInvalidValue;
        const int Pp = H / 2, Qq = W / 2;
        const long long Mll = (long long)N * Pp * Qq;
        if (Mll >= (1LL << 31)) return (int)cudaErrorInvalidValue;
        P.M = (int)Mll; P.N = Cin; P.block_n = pick_block_n(P.M, Cin, 2 * (Cout / 64));
        P.a_im2col = 1; P.PQ = Pp * Qq; P.Q = Qq; P.stride = 1; P.pad = 0; P.S = S; P.cblocks = Cout / 64; P.taps = R * S;
        P.dstride = 2; P.OH = H; P.OW = W; P.dx = (__nv_bfloat16*)dx;
        int nc = 0;
        // heaviest class first so that the long work items start early
        for (int pass = 4; pass >= 1; --pass)
            for (int a = 0; a < 2; ++a)
                for (int b = 0; b < 2; ++b) {
                    int rs[2], dps[2], nr = 0, ss[2], dqs[2], ns = 0;
                    for (int r = 0; r < R; ++r) if (((a + pad - r) & 1) == 0 && a + pad - r >= 0) { rs[nr] = r; dps[nr++] = (a + pad - r) / 2; }
                    for (int q = 0; q < S; ++q) if (((b + pad - q) & 1) == 0 && b + pad - q >= 0) { ss[ns] = q; dqs[ns++] = (b + pad - q) / 2; }
                    if (nr * ns != pass) continue;
                    P.cls_a[nc] = a; P.cls_b[nc] = b; P.cls_ntap[nc] = nr * ns;
                    for (int i = 0; i < nr; ++i)
                        for (int j = 0; j < ns; ++j) {
                            P.cls_off[nc][i * ns + j] = (unsigned char)(dqs[j] | (dps[i] << 4));
                            P.cls_wtap[nc][i * ns + j] = (unsigned char)(rs[i] * S + ss[j]);
                        }
                    ++nc;
                }
        P.ncls = nc;
        P.zero_fill = (R == 1) ? 1 : 0;
        P.num_kb = P.cls_ntap[0] * P.cblocks;
        // dY traversed with stride 1: base pixel (i, j), tap offsets 0 / +1 (a 2-tap window with one row / column of back
        // padding: lower corner 0, upper corner 0)
        ConvGeom g{N, Pp, Qq, Cout, 1, 1, 1, 0, Pp, Qq};
        if (im2col_map(&ta, dy, g, BLOCK_M)) return -2;
        tc = ta;
        return launch(DGRAD, ta, tb, tc, P, stream);
    }
    if (stride != 1) return (int)cudaErrorInvalidValue;
    const int Pp = H + 2 * pad - R + 1, Qq = W + 2 * pad - S + 1;        // dY spatial size
    const long long Mll = (long long)N * H * W;
    if (Mll >= (1LL << 31)) return (int)cudaErrorInvalidValue;
    const int M = (int)Mll;
    const bool plain = R == 1 && pad == 0 && !force_im2col;
    P.M = M; P.N = Cin; P.num_kb = R * S * (Cout / 64); P.block_n = pick_block_n(M, Cin, R * S * (Cout / 64));
    P.a_im2col = plain ? 0 : 1; P.PQ = H * W; P.Q = W; P.stride = 1; P.pad = R - 1 - pad; P.S = S; P.cblocks = Cout / 64; P.taps = R * S; P.flip = 1;
    P.dstride = 1; P.add_src = (const __nv_bfloat16*)add_src; P.add_mask = add_src ? (const unsigned char*)add_mask : nullptr; P.c_out = (__nv_bfloat16*)dx;
    if (plain) { if (v6_make_tmap_2d_bf16(&ta, (uint64_t)dy, M, Cout, (uint64_t)Cout * 2, BLOCK_M, BLOCK_K, 1)) return -2; }
    else { ConvGeom g{N, Pp, Qq, Cout, R, S, 1, R - 1 - pad, H, W}; if (im2col_map(&ta, dy, g, BLOCK_M)) return -2; }
    if (v6_make_tmap_2d_bf16(&tc, (uint64_t)dx, M, Cin, (uint64_t)Cin * 2, 32, 32, 2)) return -2;
    return launch(DGRAD, ta, tb, tc, P, stream);
}

namespace {
// The GEMM shape of a WGRAD launch and its plan (N tile, k-ranges per tile); shared by the launch and its workspace query.
int wgrad_shape(igemm::Params& P, int N, int H, int W, int Cin, int Cout, int R, int S, int stride, int pad, int splits) {
    if (Cin % 64 != 0 || Cout % 8 != 0 || (R != S && pad != 0)) return (int)cudaErrorInvalidValue;
    const int Pp = (H + 2 * pad - R) / stride + 1, Qq = (W + 2 * pad - S) / stride + 1;
    const long long pix = (long long)N * Pp * Qq;
    if (pix >= (1LL << 31)) return (int)cudaErrorInvalidValue;
    P.M = Cout; P.N = R * S * Cin; P.num_kb = (int)((pix + 63) / 64); P.block_n = 256;
    P.PQ = Pp * Qq; P.Q = Qq; P.stride = stride; P.pad = pad; P.S = S; P.cblocks = Cin / 64; P.taps = R * S;
    if (splits <= 0) {
        // (N tile, k-ranges per tile) by a small cost model in cycles: waves x k-blocks x max(MMA, operand fetch through L2) for the
        // main loop; the epilogue moves Cout x R*S*Cin x 4 B by plain load-add-store (~3000 B/cycle) when a tile has one k-range;
        // with several, each k-range stores its partial and the ordered sum reads them all back and updates dW (priced at the
        // same plain-memory rate, not measured separately).  Few tiles + long K (the
        // 56x56 layers) -> many k-ranges of a tiny output; big filters + short K (7x7 / 14x14 layers, nn.Linear) -> one k-range.
        // MEASURED while split tiles were still summed by L2 reductions (~370 B/cycle): the model's plan was slower than the simple one
        // below (about one wave of items, 256-column tiles):
        // nn.Linear 768 -> 3072 at 4096 tokens 38 vs 27 us, ResNet-50 round 51.5 vs 50.4 ms, BERT-base 31.4 vs 30.0 ms -- the
        // owned-tile load-add-store epilogue (32 rows x 16 B per instruction, 1 KB apart) and the longer per-CTA K loop cost more than
        // the reductions they avoid.  Kept behind V6B200_WGRAD_PLAN=1 with its tests.
        static const bool legacy = [] { const char* e = getenv("V6B200_WGRAD_PLAN"); return !(e && e[0] == '1'); }();
        double best = 1e30;
        int best_bn = 256, best_s = 1;
        const double out_bytes = (double)Cout * P.N * 4.0;
        for (int bn : {256, 128}) {
            const long long tiles = (long long)((Cout + 127) / 128) * ((P.N + bn - 1) / bn);
            const double per_kb = fmax(2.0 * bn, (16384.0 + bn * 128.0) / 60.0);
            for (int s = 1; s <= 64; s = s < 4 ? s + 1 : s * 2) {
                if (s > 1 && P.num_kb / s < 4) break;                    // >= 4 k-blocks per item
                const long long items = tiles * s;
                const double waves = (double)((items + 147) / 148);
                const double kb = (double)((P.num_kb + s - 1) / s);
                const double t = waves * (kb * per_kb + 1500.0) + (s == 1 ? out_bytes / 3000.0 : out_bytes * (2.0 * s + 2.0) / 3000.0);
                if (t < best) { best = t; best_bn = bn; best_s = s; }
            }
        }
        if (legacy) {
            const int tiles = ((Cout + 127) / 128) * ((P.N / 64 + 3) / 4);
            best_bn = 256;
            best_s = (148 + tiles - 1) / tiles;
            const int max_splits = P.num_kb / 4 > 0 ? P.num_kb / 4 : 1;
            if (best_s > max_splits) best_s = max_splits;
        }
        P.block_n = best_bn;
        splits = best_s;
    }
    if (splits > P.num_kb) splits = P.num_kb;
    P.kb_per_split = (P.num_kb + splits - 1) / splits;
    P.splits = (P.num_kb + P.kb_per_split - 1) / P.kb_per_split;
    return 0;
}

// dW += the partial tiles of a WGRAD with several k-ranges per tile, in a fixed order.  A block covers 256 / groups consecutive
// float4s; thread group g sums the slices g, g + groups, ... (four loads in flight) and group 0 adds the group sums in group order.
__global__ void __launch_bounds__(256) wgrad_split_sum_kernel(const float4* __restrict__ ws, float4* __restrict__ dw, long long count4,
                                                              int splits, int groups) {
    __shared__ float4 part[256];
    const int per = 256 / groups, e = threadIdx.x % per, g = threadIdx.x / per;
    auto add = [](float4& a, const float4& v) { a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w; };
    for (long long base = (long long)blockIdx.x * per; base < count4; base += (long long)gridDim.x * per) {
        const long long i = base + e;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < count4) {
            int sp = g;
            for (; sp + 3 * groups < splits; sp += 4 * groups) {
                float4 v[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) v[u] = __ldcs(ws + (long long)(sp + u * groups) * count4 + i);
#pragma unroll
                for (int u = 0; u < 4; ++u) add(acc, v[u]);
            }
            for (; sp < splits; sp += groups) add(acc, __ldcs(ws + (long long)sp * count4 + i));
        }
        part[threadIdx.x] = acc;
        __syncthreads();
        if (g == 0 && i < count4) {
            float4 sum = part[e];
            for (int k = 1; k < groups; ++k) add(sum, part[k * per + e]);
            float4 d = dw[i];
            add(d, sum);
            dw[i] = d;
        }
        __syncthreads();
    }
}
}  // namespace

// floats of workspace v6_conv_wgrad needs for this problem (0: one k-range per tile, no workspace)
extern "C" long long v6_conv_wgrad_workspace(int N, int H, int W, int Cin, int Cout, int R, int S, int stride, int pad, int splits) {
    igemm::Params P = {};
    if (wgrad_shape(P, N, H, W, Cin, Cout, R, S, stride, pad, splits)) return 0;
    return P.splits > 1 ? (long long)P.splits * P.M * P.N : 0;
}

// dw[Cout,R,S,Cin] (fp32) += scale * dy[N,P,Q,Cout]^T . im2col(x[N,H,W,Cin]); ws: v6_conv_wgrad_workspace floats (the k-range partials)
extern "C" int v6_conv_wgrad(const void* dy, const void* x, float* dw, int N, int H, int W, int Cin, int Cout, int R, int S, int stride,
                             int pad, float scale, int splits, int force_im2col, long long pitch_w, long long pitch_h, long long pitch_n,
                             float* ws, long long ws_floats, cudaStream_t stream) {
    using namespace igemm;
    Params P = {};
    const int rc = wgrad_shape(P, N, H, W, Cin, Cout, R, S, stride, pad, splits);
    if (rc) return rc;
    const long long pix = (long long)N * P.PQ;
    const bool plain = R == 1 && S == 1 && stride == 1 && pad == 0 && !force_im2col && !pitch_w;
    P.b_im2col = plain ? 0 : 1;
    P.dw = dw; P.ldw = (long long)R * S * Cin; P.out_scale = scale;
    const long long count = (long long)P.M * P.N;
    if (P.splits > 1) {
        if (ws == nullptr || ws_floats < P.splits * count) return (int)cudaErrorInvalidValue;
        P.ws = ws;
    }
    alignas(64) CUtensorMap ta, tb, tc;
    if (v6_make_tmap_2d_bf16(&ta, (uint64_t)dy, (uint64_t)pix, Cout, (uint64_t)Cout * 2, 64, 64, 1)) return -2;
    if (plain) { if (v6_make_tmap_2d_bf16(&tb, (uint64_t)x, (uint64_t)pix, Cin, (uint64_t)Cin * 2, 64, 64, 1)) return -2; }
    else { ConvGeom g{N, H, W, Cin, R, S, stride, pad, P.PQ / P.Q, P.Q, pitch_w, pitch_h, pitch_n}; if (im2col_map(&tb, x, g, 64)) return -2; }
    tc = ta;
    const int lrc = launch(WGRAD, ta, tb, tc, P, stream);
    if (lrc || P.splits == 1) return lrc;
    // enough (element, slice group) threads to fill the GPU: many slices of a small filter are summed by up to 32 groups
    const long long count4 = count / 4;                  // R*S*Cin is a multiple of 64
    int groups = 1;
    while (groups < 32 && groups * 2 <= P.splits && count4 * groups < 148LL * 2048) groups *= 2;
    const int per = 256 / groups;
    const long long blocks = (count4 + per - 1) / per;
    wgrad_split_sum_kernel<<<(unsigned)(blocks < 148 * 8 ? blocks : 148 * 8), 256, 0, stream>>>(
        reinterpret_cast<const float4*>(ws), reinterpret_cast<float4*>(dw), count4, P.splits, groups);
    V6_CHECK_LAUNCH();
    return 0;
}
