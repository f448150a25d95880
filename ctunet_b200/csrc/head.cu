// Network head: last_conv 1x1x1 + bias over the (virtual) concatenation of blocked sources, then the
// reference's output non-linearities, written as fp32 NCDHW (what the reference returns).
//   generic UNet   : lc -> [softmax] -> [sigmoid]                      models.py:255-259
//   UNetSP / UNetDO: ... -> skull = [s0, s1+s2], flap = [1-s1, s1]     models.py:319-330
//   UNetSPSmall    : ... -> softmax(skull), softmax(flap)              models.py:364-365
//   legacy         : softmax(lc)                                       models.py:535-538
// Backward recomputes lc from the sources (they are needed for dW anyway) and chains back.
#include "loss_math.cuh"

namespace ctu {

constexpr int kHeadThreads = 256;
constexpr int kHeadMaxCb = 4;

struct HeadParams {
    const void* src[CTU_MAX_SRC];
    void* dsrc[CTU_MAX_SRC];
    int src_cb[CTU_MAX_SRC];
    int nsrc;
    SrcMap m;
    const float* w;       // native [cout][c_total]
    const float* bias;
    int cout, flags;
    float* out0;
    float* out1;
    const float* dout0;
    const float* dout1;
    const float* fo0;     // forward outputs (nullable): head_bwd recovers the sigmoid values from them
    const float* fo1;
    float* dw;
    float* db;
    int n;
    long long spatial;
    // fused head + loss (ctu_head_loss_fwd / ctu_head_loss_bwd): one-hot float targets and the per-sample loss sums
    const float* tgt0;
    const float* tgt1;
    double* lsums;        // [pairs][n][4]: sum q*t, sum q*q, sum t*t, CE sum
    int tgt_u8;           // targets are uint8 class-1 masks [n][spatial] (two classes) instead of one-hot float [n][C][spatial]
    int softmax_for_dice, want_ce;
    float g_ce, g_dice;
};

// wsm[o][cbt*8]: weight of output o for (blocked, padded) input lane; pad lanes 0.
template <int CO>
__device__ __forceinline__ void load_head_weights(const HeadParams& p, float* wsm, float* bsm) {
    const int lanes = p.m.cb_total * 8;
    for (int i = threadIdx.x; i < CO * lanes; i += blockDim.x) {
        const int o = i / lanes, l = i % lanes;
        const int cib = l >> 3, ci = l & 7;
        int s = 0;
        for (int q = 1; q < CTU_MAX_SRC; ++q)
            if (q < p.m.nsrc && cib >= p.m.cboff[q]) s = q;
        const int cl = (cib - p.m.cboff[s]) * 8 + ci;
        wsm[i] = cl < p.m.ch[s] ? p.w[(long long)o * p.m.c_total + p.m.choff[s] + cl] : 0.f;
    }
    if (threadIdx.x < CO) bsm[threadIdx.x] = p.bias ? p.bias[threadIdx.x] : 0.f;
}

template <int CO> struct HeadVals {
    float lc[CO];   // logits
    float sm[CO];   // after optional softmax
    float sg[CO];   // after optional sigmoid (the plain output)
    float o0[2], o1[2];   // SP outputs (after optional pair softmax)
};

// FAST (the fused head + loss kernels only): approximate exponential / reciprocal (abs. error ~1e-7 on the outputs)
template <bool FAST> __device__ __forceinline__ float head_exp(float x) { return FAST ? __expf(x) : expf(x); }
template <bool FAST> __device__ __forceinline__ float head_div(float a, float b) { return FAST ? __fdividef(a, b) : a / b; }

template <int CO, bool FAST = false>
__device__ __forceinline__ void head_forward_chain(HeadVals<CO>& h, int flags) {
    if (flags & CTU_HEAD_SOFTMAX) {
        float mx = h.lc[0];
#pragma unroll
        for (int o = 1; o < CO; ++o) mx = fmaxf(mx, h.lc[o]);
        float sum = 0.f;
#pragma unroll
        for (int o = 0; o < CO; ++o) {
            h.sm[o] = head_exp<FAST>(h.lc[o] - mx);
            sum += h.sm[o];
        }
#pragma unroll
        for (int o = 0; o < CO; ++o) h.sm[o] = head_div<FAST>(h.sm[o], sum);
    } else {
#pragma unroll
        for (int o = 0; o < CO; ++o) h.sm[o] = h.lc[o];
    }
#pragma unroll
    for (int o = 0; o < CO; ++o)
        h.sg[o] = (flags & CTU_HEAD_SIGMOID) ? head_div<FAST>(1.f, 1.f + head_exp<FAST>(-h.sm[o])) : h.sm[o];
    if (CO == 3 && (flags & (CTU_HEAD_SP | CTU_HEAD_SP_SOFTMAX))) {
        h.o0[0] = h.sg[0];
        h.o0[1] = h.sg[1] + h.sg[CO - 1];
        h.o1[0] = 1.f - h.sg[1];
        h.o1[1] = h.sg[1];
        if (flags & CTU_HEAD_SP_SOFTMAX) {
            float m0 = fmaxf(h.o0[0], h.o0[1]);
            float e0 = head_exp<FAST>(h.o0[0] - m0), e1 = head_exp<FAST>(h.o0[1] - m0);
            h.o0[0] = head_div<FAST>(e0, e0 + e1);
            h.o0[1] = head_div<FAST>(e1, e0 + e1);
            float m1 = fmaxf(h.o1[0], h.o1[1]);
            e0 = head_exp<FAST>(h.o1[0] - m1);
            e1 = head_exp<FAST>(h.o1[1] - m1);
            h.o1[0] = head_div<FAST>(e0, e0 + e1);
            h.o1[1] = head_div<FAST>(e1, e0 + e1);
        }
    }
}

// Source of blocked input lane group c (compile-time c after unrolling keeps xs[] in registers).
__device__ __forceinline__ int head_block_source(const HeadParams& p, int c) {
    int q = 0;
#pragma unroll
    for (int qq = 1; qq < CTU_MAX_SRC; ++qq)
        if (qq < p.m.nsrc && c >= p.m.cboff[qq]) q = qq;
    return q;
}

template <typename T, int CBT>
__device__ __forceinline__ void head_load(const HeadParams& p, int n, long long s, V8 (&xs)[CBT]) {
#pragma unroll
    for (int c = 0; c < CBT; ++c) {
        const int q = head_block_source(p, c);
        const int b = c - p.m.cboff[q];
        const T* sp = reinterpret_cast<const T*>(p.src[q]);
        xs[c] = Vec8<T>::load(sp + (((long long)n * p.src_cb[q] + b) * p.spatial + s) * 8);
    }
}

template <int CO, int CBT>
__device__ __forceinline__ void head_logits_of(const float* wsm, const float* bsm, HeadVals<CO>& h, const V8 (&xs)[CBT]) {
#pragma unroll
    for (int o = 0; o < CO; ++o) h.lc[o] = bsm[o];
#pragma unroll
    for (int c = 0; c < CBT; ++c)
#pragma unroll
        for (int o = 0; o < CO; ++o)
#pragma unroll
            for (int j = 0; j < 8; ++j) h.lc[o] = fmaf(xs[c].v[j], wsm[o * CBT * 8 + c * 8 + j], h.lc[o]);
}

template <typename T, int CO, int CBT>
__device__ __forceinline__ void head_logits(const HeadParams& p, const float* wsm, const float* bsm, int n, long long s,
                                            HeadVals<CO>& h, V8 (&xs)[CBT]) {
    head_load<T, CBT>(p, n, s, xs);
    head_logits_of<CO, CBT>(wsm, bsm, h, xs);
}

template <typename T, int CO, int CBT>
__global__ void __launch_bounds__(kHeadThreads) head_fwd_kernel(HeadParams p) {
    extern __shared__ float hsm[];
    float* wsm = hsm;
    float* bsm = hsm + CO * CBT * 8;
    load_head_weights<CO>(p, wsm, bsm);
    __syncthreads();
    const long long total = (long long)p.n * p.spatial;
    const bool sp = (p.flags & (CTU_HEAD_SP | CTU_HEAD_SP_SOFTMAX)) != 0;
    if ((p.spatial & 3) == 0) {
        // four consecutive voxels per thread: 4 x CBT 16-byte loads in flight, one 16-byte store per output plane
        const long long groups = total >> 2, sg = p.spatial >> 2;
        for (long long i = (long long)blockIdx.x * kHeadThreads + threadIdx.x; i < groups; i += (long long)gridDim.x * kHeadThreads) {
            const int n = (int)(i / sg);
            const long long s = (i - (long long)n * sg) << 2;
            V8 xs[4][CBT];
#pragma unroll
            for (int v = 0; v < 4; ++v) head_load<T, CBT>(p, n, s + v, xs[v]);
            float o[4][CO > 4 ? CO : 4];
#pragma unroll
            for (int v = 0; v < 4; ++v) {
                HeadVals<CO> h;
                head_logits_of<CO, CBT>(wsm, bsm, h, xs[v]);
                head_forward_chain<CO>(h, p.flags);
                if (sp) {
                    o[v][0] = h.o0[0]; o[v][1] = h.o0[1]; o[v][2] = h.o1[0]; o[v][3] = h.o1[1];
                } else {
#pragma unroll
                    for (int c = 0; c < CO; ++c) o[v][c] = h.sg[c];
                }
            }
            if (sp) {
                *reinterpret_cast<float4*>(p.out0 + ((long long)n * 2 + 0) * p.spatial + s) = make_float4(o[0][0], o[1][0], o[2][0], o[3][0]);
                *reinterpret_cast<float4*>(p.out0 + ((long long)n * 2 + 1) * p.spatial + s) = make_float4(o[0][1], o[1][1], o[2][1], o[3][1]);
                *reinterpret_cast<float4*>(p.out1 + ((long long)n * 2 + 0) * p.spatial + s) = make_float4(o[0][2], o[1][2], o[2][2], o[3][2]);
                *reinterpret_cast<float4*>(p.out1 + ((long long)n * 2 + 1) * p.spatial + s) = make_float4(o[0][3], o[1][3], o[2][3], o[3][3]);
            } else {
#pragma unroll
                for (int c = 0; c < CO; ++c)
                    *reinterpret_cast<float4*>(p.out0 + ((long long)n * CO + c) * p.spatial + s) = make_float4(o[0][c], o[1][c], o[2][c], o[3][c]);
            }
        }
        return;
    }
    for (long long i = (long long)blockIdx.x * kHeadThreads + threadIdx.x; i < total; i += (long long)gridDim.x * kHeadThreads) {
        const int n = (int)(i / p.spatial);
        const long long s = i % p.spatial;
        HeadVals<CO> h;
        V8 xs[CBT];
        head_logits<T, CO, CBT>(p, wsm, bsm, n, s, h, xs);
        head_forward_chain<CO>(h, p.flags);
        if (sp) {
            p.out0[((long long)n * 2 + 0) * p.spatial + s] = h.o0[0];
            p.out0[((long long)n * 2 + 1) * p.spatial + s] = h.o0[1];
            p.out1[((long long)n * 2 + 0) * p.spatial + s] = h.o1[0];
            p.out1[((long long)n * 2 + 1) * p.spatial + s] = h.o1[1];
        } else {
#pragma unroll
            for (int o = 0; o < CO; ++o) p.out0[((long long)n * CO + o) * p.spatial + s] = h.sg[o];
        }
    }
}

// PART 0: source gradients and parameter gradients; 1: source gradients only (the critical path of the backward
// pass); 2: parameter gradients only (a leaf: the engine runs it beside the weight gradients).  The 48+ per-thread
// dW accumulators are what limits occupancy, so the split halves the latency of the part the decoder waits for.
// FROMOUT (plain-sigmoid SP head, CO == 3): the sigmoid values are recovered from the forward OUTPUTS
// (skull = [s0, s1+s2], flap = [1-s1, s1]) instead of being recomputed from the inputs: the source-gradient launch then
// reads 28 B and writes 32 B per voxel, with no logits and no exponentials.
template <typename T, int CO, int CBT, int PART, bool FROMOUT>
__global__ void __launch_bounds__(kHeadThreads) head_bwd_kernel(HeadParams p) {
    extern __shared__ float hsm[];
    float* wsm = hsm;
    float* bsm = hsm + CO * CBT * 8;
    float* red = bsm + 8;                           // [8 warps][CO*CBT*8 + CO]
    load_head_weights<CO>(p, wsm, bsm);
    __syncthreads();
    const long long total = (long long)p.n * p.spatial;
    const bool sp = (p.flags & (CTU_HEAD_SP | CTU_HEAD_SP_SOFTMAX)) != 0;
    float gw[CO][CBT * 8], gb[CO];
#pragma unroll
    for (int o = 0; o < CO; ++o) {
        gb[o] = 0.f;
#pragma unroll
        for (int l = 0; l < CBT * 8; ++l) gw[o][l] = 0.f;
    }
    // software pipeline: the inputs of the next voxel are in flight while the current one is processed
    const long long stride = (long long)gridDim.x * kHeadThreads;
    long long i = (long long)blockIdx.x * kHeadThreads + threadIdx.x;
    V8 xn[CBT];
    float gn[4] = {0.f, 0.f, 0.f, 0.f}, on[3] = {0.f, 0.f, 0.f};
    constexpr bool NEEDX = !FROMOUT || PART != 1;
    auto fetch = [&](long long idx, V8 (&xo)[CBT], float (&go)[4], float (&oo)[3]) {
        const int n = (int)(idx / p.spatial);
        const long long s = idx % p.spatial;
        if (NEEDX) head_load<T, CBT>(p, n, s, xo);
        if (FROMOUT) {
            oo[0] = p.fo0[((long long)n * 2 + 0) * p.spatial + s];
            oo[1] = p.fo0[((long long)n * 2 + 1) * p.spatial + s];
            oo[2] = p.fo1[((long long)n * 2 + 1) * p.spatial + s];
        }
        if (sp) {
            go[0] = p.dout0 ? p.dout0[((long long)n * 2 + 0) * p.spatial + s] : 0.f;
            go[1] = p.dout0 ? p.dout0[((long long)n * 2 + 1) * p.spatial + s] : 0.f;
            go[2] = p.dout1 ? p.dout1[((long long)n * 2 + 0) * p.spatial + s] : 0.f;
            go[3] = p.dout1 ? p.dout1[((long long)n * 2 + 1) * p.spatial + s] : 0.f;
        } else {
#pragma unroll
            for (int o = 0; o < CO; ++o) go[o] = p.dout0[((long long)n * CO + o) * p.spatial + s];
        }
    };
    if (i < total) fetch(i, xn, gn, on);
    for (; i < total; i += stride) {
        const int n = (int)(i / p.spatial);
        const long long s = i % p.spatial;
        V8 xs[CBT];
        float gc[4], oc[3];
#pragma unroll
        for (int c = 0; c < CBT; ++c) xs[c] = xn[c];
#pragma unroll
        for (int o = 0; o < 4; ++o) gc[o] = gn[o];
#pragma unroll
        for (int o = 0; o < 3; ++o) oc[o] = on[o];
        if (i + stride < total) fetch(i + stride, xn, gn, on);
        HeadVals<CO> h;
        if (FROMOUT) {
            h.sg[0] = oc[0];
            h.sg[1] = oc[2];
            h.sg[CO - 1] = oc[1] - oc[2];
        } else {
            head_logits_of<CO, CBT>(wsm, bsm, h, xs);
            head_forward_chain<CO>(h, p.flags);
        }
        float dsg[CO];
        if (sp) {
            float g00 = gc[0], g01 = gc[1], g10 = gc[2], g11 = gc[3];
            if (p.flags & CTU_HEAD_SP_SOFTMAX) {
                // out = softmax(pair): d(pair_j) = out_j * (g_j - sum_i g_i out_i)
                float d0 = g00 * h.o0[0] + g01 * h.o0[1];
                g00 = h.o0[0] * (g00 - d0);
                g01 = h.o0[1] * (g01 - d0);
                float d1 = g10 * h.o1[0] + g11 * h.o1[1];
                g10 = h.o1[0] * (g10 - d1);
                g11 = h.o1[1] * (g11 - d1);
            }
            // skull = [s0, s1+s2], flap = [1-s1, s1]
            dsg[0] = g00;
            dsg[1] = g01 - g10 + g11;
            dsg[CO - 1] = g01;
        } else {
#pragma unroll
            for (int o = 0; o < CO; ++o) dsg[o] = gc[o];
        }
        float dsm[CO], dlc[CO];
#pragma unroll
        for (int o = 0; o < CO; ++o) dsm[o] = (p.flags & CTU_HEAD_SIGMOID) ? dsg[o] * h.sg[o] * (1.f - h.sg[o]) : dsg[o];
        if (p.flags & CTU_HEAD_SOFTMAX) {
            float dot = 0.f;
#pragma unroll
            for (int o = 0; o < CO; ++o) dot += dsm[o] * h.sm[o];
#pragma unroll
            for (int o = 0; o < CO; ++o) dlc[o] = h.sm[o] * (dsm[o] - dot);
        } else {
#pragma unroll
            for (int o = 0; o < CO; ++o) dlc[o] = dsm[o];
        }
        // parameter gradients (per-thread partials) and source gradients
        if (PART != 2) {
#pragma unroll
        for (int c = 0; c < CBT; ++c) {
            const int q = head_block_source(p, c);
            const int b = c - p.m.cboff[q];
            T* dp = reinterpret_cast<T*>(p.dsrc[q]);
            V8 g;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                float a = 0.f;
#pragma unroll
                for (int o = 0; o < CO; ++o) a = fmaf(dlc[o], wsm[o * CBT * 8 + c * 8 + j], a);
                g.v[j] = a;
            }
            if (dp != nullptr) Vec8<T>::store(dp + (((long long)n * p.src_cb[q] + b) * p.spatial + s) * 8, g);
        }
        }
        if (PART != 1) {
#pragma unroll
        for (int o = 0; o < CO; ++o) {
            gb[o] += dlc[o];
#pragma unroll
            for (int c = 0; c < CBT; ++c)
#pragma unroll
                for (int j = 0; j < 8; ++j) gw[o][c * 8 + j] = fmaf(dlc[o], xs[c].v[j], gw[o][c * 8 + j]);
        }
        }
    }
    if (PART == 1) return;
    // block reduction of the CO*(CBT*8+1) partials, then one atomic each
    constexpr int NV = CO * CBT * 8 + CO;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 0; o < CO; ++o) {
#pragma unroll
        for (int l = 0; l < CBT * 8; ++l) {
            float v = warp_sum(gw[o][l]);
            if (lane == 0) red[warp * NV + o * CBT * 8 + l] = v;
        }
        float v = warp_sum(gb[o]);
        if (lane == 0) red[warp * NV + CO * CBT * 8 + o] = v;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < NV; i += kHeadThreads) {
        float v = 0.f;
        for (int wq = 0; wq < kHeadThreads / 32; ++wq) v += red[wq * NV + i];
        if (i < CO * CBT * 8) {
            const int o = i / (CBT * 8), l = i % (CBT * 8);
            const int cib = l >> 3, ci = l & 7;
            int s = 0;
            for (int q = 1; q < CTU_MAX_SRC; ++q)
                if (q < p.m.nsrc && cib >= p.m.cboff[q]) s = q;
            const int cl = (cib - p.m.cboff[s]) * 8 + ci;
            if (cl < p.m.ch[s]) atomicAdd(p.dw + (long long)o * p.m.c_total + p.m.choff[s] + cl, v);
        } else {
            atomicAdd(p.db + (i - CO * CBT * 8), v);
        }
    }
}

static int head_setup(HeadParams& p, const void* const* h_srcs, const int* h_src_channels, int nsrc, const float* w,
                      const float* bias, int cout, int flags, int n, long long spatial, const char* what) {
    int rc = make_srcmap(p.m, nsrc, h_src_channels);
    if (rc != CTU_OK) return rc;
    CTU_REQUIRE(h_srcs && w && cout >= 1 && cout <= 4 && n > 0 && spatial > 0, "%s: bad arguments (cout must be 1..4)", what);
    CTU_REQUIRE(p.m.cb_total <= kHeadMaxCb, "%s: at most %d input blocks supported (got %d)", what, kHeadMaxCb, p.m.cb_total);
    if (flags & (CTU_HEAD_SP | CTU_HEAD_SP_SOFTMAX)) CTU_REQUIRE(cout == 3, "%s: the SP head needs 3 output channels", what);
    for (int i = 0; i < CTU_MAX_SRC; ++i) {
        p.src[i] = i < nsrc ? h_srcs[i] : nullptr;
        p.dsrc[i] = nullptr;
        p.src_cb[i] = i < nsrc ? (p.m.ch[i] + 7) / 8 : 0;
        if (i < nsrc) CTU_REQUIRE(h_srcs[i] != nullptr, "%s: null source %d", what, i);
    }
    p.nsrc = nsrc; p.w = w; p.bias = bias; p.cout = cout; p.flags = flags; p.n = n; p.spatial = spatial;
    return CTU_OK;
}

static int head_grid(long long total) {
    long long g = (total + kHeadThreads - 1) / kHeadThreads;
    const long long cap = 148 * 8;
    return (int)(g < cap ? g : cap);
}

template <typename T, int CO>
static int head_fwd_launch(const HeadParams& p, int grid, size_t smem, cudaStream_t stream) {
    switch (p.m.cb_total) {
        case 1: head_fwd_kernel<T, CO, 1><<<grid, kHeadThreads, smem, stream>>>(p); break;
        case 2: head_fwd_kernel<T, CO, 2><<<grid, kHeadThreads, smem, stream>>>(p); break;
        case 3: head_fwd_kernel<T, CO, 3><<<grid, kHeadThreads, smem, stream>>>(p); break;
        default: head_fwd_kernel<T, CO, 4><<<grid, kHeadThreads, smem, stream>>>(p); break;
    }
    return check_launch("ctu_head_fwd");
}

template <typename T, int CO, int PART>
static int head_bwd_launch_part(const HeadParams& p, cudaStream_t stream) {
    const int cbt = p.m.cb_total;
    const int nv = CO * cbt * 8 + CO;
    const size_t smem = (size_t)(CO * cbt * 8 + 8 + (kHeadThreads / 32) * nv) * sizeof(float);
    int grid = head_grid((long long)p.n * p.spatial);
    if (PART != 1 && grid > 148 * 2) grid = 148 * 2;   // every block ends with CO*(Cin+1) same-address atomics
    const bool fromout = CO == 3 && p.fo0 != nullptr && p.fo1 != nullptr &&
                         p.flags == (CTU_HEAD_SIGMOID | CTU_HEAD_SP);
    if (fromout) {
        if (CO == 3) {       // (compile-time guard: the fast path is only instantiated for the 3-channel SP head)
            constexpr int C3 = CO == 3 ? 3 : 1;
            switch (cbt) {
                case 1: head_bwd_kernel<T, C3, 1, PART, CO == 3><<<grid, kHeadThreads, smem, stream>>>(p); break;
                case 2: head_bwd_kernel<T, C3, 2, PART, CO == 3><<<grid, kHeadThreads, smem, stream>>>(p); break;
                case 3: head_bwd_kernel<T, C3, 3, PART, CO == 3><<<grid, kHeadThreads, smem, stream>>>(p); break;
                default: head_bwd_kernel<T, C3, 4, PART, CO == 3><<<grid, kHeadThreads, smem, stream>>>(p); break;
            }
        }
        return check_launch("ctu_head_bwd");
    }
    switch (cbt) {
        case 1: head_bwd_kernel<T, CO, 1, PART, false><<<grid, kHeadThreads, smem, stream>>>(p); break;
        case 2: head_bwd_kernel<T, CO, 2, PART, false><<<grid, kHeadThreads, smem, stream>>>(p); break;
        case 3: head_bwd_kernel<T, CO, 3, PART, false><<<grid, kHeadThreads, smem, stream>>>(p); break;
        default: head_bwd_kernel<T, CO, 4, PART, false><<<grid, kHeadThreads, smem, stream>>>(p); break;
    }
    return check_launch("ctu_head_bwd");
}

template <typename T, int CO>
static int head_bwd_launch(const HeadParams& p, int part, cudaStream_t stream) {
    if (part == 1) return head_bwd_launch_part<T, CO, 1>(p, stream);
    if (part == 2) return head_bwd_launch_part<T, CO, 2>(p, stream);
    return head_bwd_launch_part<T, CO, 0>(p, stream);
}


// ------------------------------------------------------------------------------------------------ fused head + loss
// The training step never needs the network outputs themselves -- only the loss sums and, in the backward pass, the
// gradient with respect to the head's inputs.  The fused kernels recompute the head (14 multiply-adds per output) from
// the blocked sources and feed the loss arithmetic of loss_math.cuh in registers: the two fp32 [B,2,D,H,W] outputs and
// their gradients (64 B per voxel, written once and read twice each) never touch HBM.
//   forward : reads 16 B per source block + the one-hot targets, accumulates the per-sample sums (grid.y = sample)
//   backward: the same reads, writes the source gradients (PART 1) / reduces the parameter gradients (PART 2)
// PAIRS = 2: the SP heads (outputs skull = o0, flap = o1, two classes each; ProblemHandler.py:228-298);
// PAIRS = 1: the plain head with CO classes against one target (ProblemHandler.py:59-91).
// Two x-adjacent voxels of the targets of one pair: one-hot float planes, or a uint8 class-1 mask (t = [1 - m, m]).
template <int C, bool U8>
__device__ __forceinline__ void head_load_targets2(const float* tf, long long spatial, int n, long long s, float (&t)[C][2]) {
    if (U8) {
        const unsigned char* m = reinterpret_cast<const unsigned char*>(tf) + (long long)n * spatial + s;
        const uchar2 v = *reinterpret_cast<const uchar2*>(m);
        const float a = v.x ? 1.f : 0.f, b = v.y ? 1.f : 0.f;
        t[0][0] = 1.f - a; t[0][1] = 1.f - b;
        t[C - 1][0] = a; t[C - 1][1] = b;
    } else {
        const float* base = tf + (long long)n * C * spatial + s;
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const float2 v = __ldg(reinterpret_cast<const float2*>(base + c * spatial));
            t[c][0] = v.x; t[c][1] = v.y;
        }
    }
}
template <int C, bool U8>
__device__ __forceinline__ void head_load_targets1(const float* tf, long long spatial, int n, long long s, float (&t)[C]) {
    if (U8) {
        const float a = reinterpret_cast<const unsigned char*>(tf)[(long long)n * spatial + s] ? 1.f : 0.f;
        t[0] = 1.f - a;
        t[C - 1] = a;
    } else {
#pragma unroll
        for (int c = 0; c < C; ++c) t[c] = __ldg(tf + ((long long)n * C + c) * spatial + s);
    }
}

template <typename T, int CO, int CBT, int PAIRS, bool TU8>
__global__ void __launch_bounds__(kHeadThreads, 2) head_loss_fwd_kernel(HeadParams p) {
    extern __shared__ float hsm[];
    float* wsm = hsm;
    float* bsm = hsm + CO * CBT * 8;
    load_head_weights<CO>(p, wsm, bsm);
    __syncthreads();
    constexpr int C = PAIRS == 2 ? 2 : CO;
    const int n = blockIdx.y;
    float acc[PAIRS][4];
#pragma unroll
    for (int q = 0; q < PAIRS; ++q)
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[q][i] = 0.f;
    auto voxel = [&](const V8 (&xs)[CBT], const float (&ta)[C], const float (&tb)[C]) {
        HeadVals<CO> h;
        head_logits_of<CO, CBT>(wsm, bsm, h, xs);
        head_forward_chain<CO, true>(h, p.flags);
        if (PAIRS == 2) {
            loss_voxel_fwd2(h.o0[0], h.o0[1], ta[0], ta[C - 1], p.softmax_for_dice, p.want_ce, acc[0]);
            loss_voxel_fwd2(h.o1[0], h.o1[1], tb[0], tb[C - 1], p.softmax_for_dice, p.want_ce, acc[PAIRS - 1]);
        } else if (C == 2) {
            loss_voxel_fwd2(h.sg[0], h.sg[CO - 1], ta[0], ta[C - 1], p.softmax_for_dice, p.want_ce, acc[0]);
        } else {
            float x[C];
#pragma unroll
            for (int c = 0; c < C; ++c) x[c] = h.sg[c < CO ? c : 0];
            loss_voxel_fwd<C>(x, ta, p.softmax_for_dice, p.want_ce, acc[0]);
        }
    };
    if ((p.spatial & 1) == 0) {
        // two x-adjacent voxels per thread and iteration: 2 x CBT 16-byte source loads + 8-byte target loads in flight
        const long long groups = p.spatial >> 1;
        for (long long gi = (long long)blockIdx.x * kHeadThreads + threadIdx.x; gi < groups; gi += (long long)gridDim.x * kHeadThreads) {
            const long long s = gi << 1;
            V8 xs[2][CBT];
#pragma unroll
            for (int v = 0; v < 2; ++v) head_load<T, CBT>(p, n, s + v, xs[v]);
            float ta[C][2], tb[C][2];
#pragma unroll
            for (int c = 0; c < C; ++c) ta[c][0] = ta[c][1] = tb[c][0] = tb[c][1] = 0.f;
            head_load_targets2<C, TU8>(p.tgt0, p.spatial, n, s, ta);
            if (PAIRS == 2) head_load_targets2<C, TU8>(p.tgt1, p.spatial, n, s, tb);
#pragma unroll
            for (int v = 0; v < 2; ++v) {
                float ua[C], ub[C];
#pragma unroll
                for (int c = 0; c < C; ++c) ua[c] = ta[c][v], ub[c] = tb[c][v];
                voxel(xs[v], ua, ub);
            }
        }
    } else {
        for (long long s = (long long)blockIdx.x * kHeadThreads + threadIdx.x; s < p.spatial; s += (long long)gridDim.x * kHeadThreads) {
            V8 xs[CBT];
            head_load<T, CBT>(p, n, s, xs);
            float ua[C], ub[C];
#pragma unroll
            for (int c = 0; c < C; ++c) ua[c] = ub[c] = 0.f;
            head_load_targets1<C, TU8>(p.tgt0, p.spatial, n, s, ua);
            if (PAIRS == 2) head_load_targets1<C, TU8>(p.tgt1, p.spatial, n, s, ub);
            voxel(xs, ua, ub);
        }
    }
    __shared__ float red[kHeadThreads / 32][PAIRS * 4];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int q = 0; q < PAIRS; ++q)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float v = warp_sum(acc[q][i]);
            if (lane == 0) red[warp][q * 4 + i] = v;
        }
    __syncthreads();
    if (threadIdx.x < PAIRS * 4) {
        double v = 0.0;
        for (int wq = 0; wq < kHeadThreads / 32; ++wq) v += (double)red[wq][threadIdx.x];
        const int q = threadIdx.x >> 2, i = threadIdx.x & 3;
        atomicAdd(p.lsums + ((long long)q * p.n + n) * 4 + i, v);
    }
}

// comps = [ce_lambda * CE per pair] + [dice_lambda * Dice per pair] + [total], the order of ProblemHandler.py:241-298
__global__ void head_loss_finalize_kernel(const double* __restrict__ sums, int pairs, int nb, long long spatial, float ce_lambda,
                                          float dice_lambda, float* __restrict__ comps, float* __restrict__ mirror) {
    const double eps = 0.0000001;
    float ce[2], dice[2];
    for (int q = 0; q < pairs; ++q) {
        double dsum = 0.0, c = 0.0;
        for (int i = 0; i < nb; ++i) {
            const double* s4 = sums + ((long long)q * nb + i) * 4;
            dsum += (s4[0] + eps) / (s4[1] + s4[2] + eps);
            c += s4[3];
        }
        ce[q] = (float)(c / ((double)nb * (double)spatial));
        dice[q] = (float)(1.0 - 2.0 * dsum / (double)nb);
    }
    int k = 0;
    float total = 0.f;
    if (ce_lambda != 0.f)
        for (int q = 0; q < pairs; ++q, ++k) {
            comps[k] = ce_lambda * ce[q];
            total = k == 0 ? comps[k] : total + comps[k];
        }
    if (dice_lambda != 0.f)
        for (int q = 0; q < pairs; ++q, ++k) {
            comps[k] = dice_lambda * dice[q];
            total = k == 0 ? comps[k] : total + comps[k];
        }
    comps[k] = total;
    if (mirror)
        for (int i = 0; i <= k; ++i) mirror[i] = comps[i];
}

// Source gradients; the logit gradients dlc [n][CO][spatial] (fp32 planes) are stored for head_param_grad_kernel, so the
// parameter-gradient launch (a leaf of the backward pass, second stream) is pure multiply-add streaming.
template <typename T, int CO, int CBT, int PAIRS, bool TU8>
__global__ void __launch_bounds__(kHeadThreads, 2) head_loss_bwd_kernel(HeadParams p) {
    extern __shared__ float hsm[];
    float* wsm = hsm;
    float* bsm = hsm + CO * CBT * 8;
    load_head_weights<CO>(p, wsm, bsm);
    __syncthreads();
    constexpr int C = PAIRS == 2 ? 2 : CO;
    const int n = blockIdx.y;
    float kt[PAIRS], kq[PAIRS];
#pragma unroll
    for (int q = 0; q < PAIRS; ++q) dice_coefficients(p.lsums + ((long long)q * p.n + n) * 4, p.n, p.g_dice, kt[q], kq[q]);
    const float kce = p.want_ce ? p.g_ce / ((float)p.n * (float)p.spatial) : 0.f;
    float* dlc_out = p.out0 + (long long)n * CO * p.spatial;       // (out0 doubles as the dlc buffer in this kernel)
    auto voxel = [&](const V8 (&xs)[CBT], const float (&ta)[C], const float (&tb)[C], long long s, float (&dlc)[CO]) {
        HeadVals<CO> h;
        head_logits_of<CO, CBT>(wsm, bsm, h, xs);
        head_forward_chain<CO, true>(h, p.flags);
        float dsg[CO];
        if (PAIRS == 2) {
            float g00, g01, g10, g11;
            loss_voxel_bwd2(h.o0[0], h.o0[1], ta[0], ta[C - 1], p.softmax_for_dice, p.want_ce, kt[0], kq[0], kce, g00, g01);
            loss_voxel_bwd2(h.o1[0], h.o1[1], tb[0], tb[C - 1], p.softmax_for_dice, p.want_ce, kt[PAIRS - 1], kq[PAIRS - 1], kce,
                            g10, g11);
            if (p.flags & CTU_HEAD_SP_SOFTMAX) {
                float d0 = g00 * h.o0[0] + g01 * h.o0[1];
                g00 = h.o0[0] * (g00 - d0);
                g01 = h.o0[1] * (g01 - d0);
                float d1 = g10 * h.o1[0] + g11 * h.o1[1];
                g10 = h.o1[0] * (g10 - d1);
                g11 = h.o1[1] * (g11 - d1);
            }
            dsg[0] = g00;
            dsg[CO > 1 ? 1 : 0] = g01 - g10 + g11;
            dsg[CO - 1] = g01;
        } else if (C == 2) {
            loss_voxel_bwd2(h.sg[0], h.sg[CO - 1], ta[0], ta[C - 1], p.softmax_for_dice, p.want_ce, kt[0], kq[0], kce, dsg[0],
                            dsg[CO - 1]);
        } else {
            float x[C], gx[C];
#pragma unroll
            for (int c = 0; c < C; ++c) x[c] = h.sg[c < CO ? c : 0];
            loss_voxel_bwd<C>(x, ta, p.softmax_for_dice, p.want_ce, kt[0], kq[0], kce, gx);
#pragma unroll
            for (int o = 0; o < CO; ++o) dsg[o] = gx[o < C ? o : 0];
        }
        float dsm[CO];
#pragma unroll
        for (int o = 0; o < CO; ++o) dsm[o] = (p.flags & CTU_HEAD_SIGMOID) ? dsg[o] * h.sg[o] * (1.f - h.sg[o]) : dsg[o];
        if (p.flags & CTU_HEAD_SOFTMAX) {
            float dot = 0.f;
#pragma unroll
            for (int o = 0; o < CO; ++o) dot += dsm[o] * h.sm[o];
#pragma unroll
            for (int o = 0; o < CO; ++o) dlc[o] = h.sm[o] * (dsm[o] - dot);
        } else {
#pragma unroll
            for (int o = 0; o < CO; ++o) dlc[o] = dsm[o];
        }
#pragma unroll
        for (int c = 0; c < CBT; ++c) {
            const int q = head_block_source(p, c);
            const int b = c - p.m.cboff[q];
            T* dp = reinterpret_cast<T*>(p.dsrc[q]);
            V8 g;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                float a = 0.f;
#pragma unroll
                for (int o = 0; o < CO; ++o) a = fmaf(dlc[o], wsm[o * CBT * 8 + c * 8 + j], a);
                g.v[j] = a;
            }
            if (dp != nullptr) Vec8<T>::store(dp + (((long long)n * p.src_cb[q] + b) * p.spatial + s) * 8, g);
        }
    };
    if ((p.spatial & 1) == 0) {
        const long long groups = p.spatial >> 1;
        for (long long gi = (long long)blockIdx.x * kHeadThreads + threadIdx.x; gi < groups; gi += (long long)gridDim.x * kHeadThreads) {
            const long long s = gi << 1;
            V8 xs[2][CBT];
#pragma unroll
            for (int v = 0; v < 2; ++v) head_load<T, CBT>(p, n, s + v, xs[v]);
            float ta[C][2], tb[C][2];
#pragma unroll
            for (int c = 0; c < C; ++c) ta[c][0] = ta[c][1] = tb[c][0] = tb[c][1] = 0.f;
            head_load_targets2<C, TU8>(p.tgt0, p.spatial, n, s, ta);
            if (PAIRS == 2) head_load_targets2<C, TU8>(p.tgt1, p.spatial, n, s, tb);
            float dl[2][CO];
#pragma unroll
            for (int v = 0; v < 2; ++v) {
                float ua[C], ub[C];
#pragma unroll
                for (int c = 0; c < C; ++c) ua[c] = ta[c][v], ub[c] = tb[c][v];
                voxel(xs[v], ua, ub, s + v, dl[v]);
            }
#pragma unroll
            for (int o = 0; o < CO; ++o)
                *reinterpret_cast<float2*>(dlc_out + o * p.spatial + s) = make_float2(dl[0][o], dl[1][o]);
        }
    } else {
        for (long long s = (long long)blockIdx.x * kHeadThreads + threadIdx.x; s < p.spatial; s += (long long)gridDim.x * kHeadThreads) {
            V8 xs[CBT];
            head_load<T, CBT>(p, n, s, xs);
            float ua[C], ub[C], dl[CO];
#pragma unroll
            for (int c = 0; c < C; ++c) ua[c] = ub[c] = 0.f;
            head_load_targets1<C, TU8>(p.tgt0, p.spatial, n, s, ua);
            if (PAIRS == 2) head_load_targets1<C, TU8>(p.tgt1, p.spatial, n, s, ub);
            voxel(xs, ua, ub, s, dl);
#pragma unroll
            for (int o = 0; o < CO; ++o) dlc_out[o * p.spatial + s] = dl[o];
        }
    }
}

// dW[o][c] = sum_voxels dlc[o] * x[c], db[o] = sum_voxels dlc[o] from the stored logit gradients
template <typename T, int CO, int CBT>
__global__ void __launch_bounds__(kHeadThreads) head_param_grad_kernel(HeadParams p) {
    extern __shared__ float hsm[];
    float* red = hsm;                               // [8 warps][CO*CBT*8 + CO]
    float gw[CO][CBT * 8], gb[CO];
#pragma unroll
    for (int o = 0; o < CO; ++o) {
        gb[o] = 0.f;
#pragma unroll
        for (int l = 0; l < CBT * 8; ++l) gw[o][l] = 0.f;
    }
    const long long total = (long long)p.n * p.spatial;
    for (long long i = (long long)blockIdx.x * kHeadThreads + threadIdx.x; i < total; i += (long long)gridDim.x * kHeadThreads) {
        const int n = (int)(i / p.spatial);
        const long long s = i - (long long)n * p.spatial;
        V8 xs[CBT];
        head_load<T, CBT>(p, n, s, xs);
        float dlc[CO];
#pragma unroll
        for (int o = 0; o < CO; ++o) dlc[o] = __ldg(p.dout0 + ((long long)n * CO + o) * p.spatial + s);
#pragma unroll
        for (int o = 0; o < CO; ++o) {
            gb[o] += dlc[o];
#pragma unroll
            for (int c = 0; c < CBT; ++c)
#pragma unroll
                for (int j = 0; j < 8; ++j) gw[o][c * 8 + j] = fmaf(dlc[o], xs[c].v[j], gw[o][c * 8 + j]);
        }
    }
    constexpr int NV = CO * CBT * 8 + CO;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 0; o < CO; ++o) {
#pragma unroll
        for (int l = 0; l < CBT * 8; ++l) {
            float v = warp_sum(gw[o][l]);
            if (lane == 0) red[warp * NV + o * CBT * 8 + l] = v;
        }
        float v = warp_sum(gb[o]);
        if (lane == 0) red[warp * NV + CO * CBT * 8 + o] = v;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < NV; i += kHeadThreads) {
        float v = 0.f;
        for (int wq = 0; wq < kHeadThreads / 32; ++wq) v += red[wq * NV + i];
        if (i < CO * CBT * 8) {
            const int o = i / (CBT * 8), l = i % (CBT * 8);
            const int cib = l >> 3, ci = l & 7;
            int sq = 0;
            for (int q = 1; q < CTU_MAX_SRC; ++q)
                if (q < p.m.nsrc && cib >= p.m.cboff[q]) sq = q;
            const int cl = (cib - p.m.cboff[sq]) * 8 + ci;
            if (cl < p.m.ch[sq]) atomicAdd(p.dw + (long long)o * p.m.c_total + p.m.choff[sq] + cl, v);
        } else {
            atomicAdd(p.db + (i - CO * CBT * 8), v);
        }
    }
}

template <typename T, int CO, int PAIRS>
static int head_loss_fwd_launch(const HeadParams& p, cudaStream_t stream) {
    const size_t smem = (size_t)(CO * p.m.cb_total * 8 + 8) * sizeof(float);
    const long long per = ((p.spatial & 1) == 0 ? p.spatial >> 1 : p.spatial);
    long long gx = (per + kHeadThreads - 1) / kHeadThreads;
    const long long cap = (148 * 16 + p.n - 1) / p.n;
    if (gx > cap) gx = cap;
    dim3 grid((unsigned)gx, p.n);
    switch (p.m.cb_total) {
        case 1: if (p.tgt_u8) head_loss_fwd_kernel<T, CO, 1, PAIRS, true><<<grid, kHeadThreads, smem, stream>>>(p); else head_loss_fwd_kernel<T, CO, 1, PAIRS, false><<<grid, kHeadThreads, smem, stream>>>(p); break;
        case 2: if (p.tgt_u8) head_loss_fwd_kernel<T, CO, 2, PAIRS, true><<<grid, kHeadThreads, smem, stream>>>(p); else head_loss_fwd_kernel<T, CO, 2, PAIRS, false><<<grid, kHeadThreads, smem, stream>>>(p); break;
        case 3: if (p.tgt_u8) head_loss_fwd_kernel<T, CO, 3, PAIRS, true><<<grid, kHeadThreads, smem, stream>>>(p); else head_loss_fwd_kernel<T, CO, 3, PAIRS, false><<<grid, kHeadThreads, smem, stream>>>(p); break;
        default: if (p.tgt_u8) head_loss_fwd_kernel<T, CO, 4, PAIRS, true><<<grid, kHeadThreads, smem, stream>>>(p); else head_loss_fwd_kernel<T, CO, 4, PAIRS, false><<<grid, kHeadThreads, smem, stream>>>(p); break;
    }
    return check_launch("ctu_head_loss_fwd");
}

template <typename T, int CO, int PAIRS>
static int head_loss_bwd_launch(const HeadParams& p, cudaStream_t stream) {
    const int cbt = p.m.cb_total;
    const size_t smem = (size_t)(CO * cbt * 8 + 8) * sizeof(float);
    const long long per = ((p.spatial & 1) == 0 ? p.spatial >> 1 : p.spatial);
    long long gx = (per + kHeadThreads - 1) / kHeadThreads;
    const long long cap = (148 * 16 + p.n - 1) / p.n;
    if (gx > cap) gx = cap;
    dim3 grid((unsigned)gx, p.n);
    switch (cbt) {
        case 1: if (p.tgt_u8) head_loss_bwd_kernel<T, CO, 1, PAIRS, true><<<grid, kHeadThreads, smem, stream>>>(p); else head_loss_bwd_kernel<T, CO, 1, PAIRS, false><<<grid, kHeadThreads, smem, stream>>>(p); break;
        case 2: if (p.tgt_u8) head_loss_bwd_kernel<T, CO, 2, PAIRS, true><<<grid, kHeadThreads, smem, stream>>>(p); else head_loss_bwd_kernel<T, CO, 2, PAIRS, false><<<grid, kHeadThreads, smem, stream>>>(p); break;
        case 3: if (p.tgt_u8) head_loss_bwd_kernel<T, CO, 3, PAIRS, true><<<grid, kHeadThreads, smem, stream>>>(p); else head_loss_bwd_kernel<T, CO, 3, PAIRS, false><<<grid, kHeadThreads, smem, stream>>>(p); break;
        default: if (p.tgt_u8) head_loss_bwd_kernel<T, CO, 4, PAIRS, true><<<grid, kHeadThreads, smem, stream>>>(p); else head_loss_bwd_kernel<T, CO, 4, PAIRS, false><<<grid, kHeadThreads, smem, stream>>>(p); break;
    }
    return check_launch("ctu_head_loss_bwd");
}

template <typename T, int CO>
static int head_param_grad_launch(const HeadParams& p, cudaStream_t stream) {
    const int cbt = p.m.cb_total;
    const int nv = CO * cbt * 8 + CO;
    const size_t smem = (size_t)((kHeadThreads / 32) * nv) * sizeof(float);
    int grid = head_grid((long long)p.n * p.spatial);
    if (grid > 148 * 2) grid = 148 * 2;          // every block ends with CO*(Cin+1) same-address atomics
    switch (cbt) {
        case 1: head_param_grad_kernel<T, CO, 1><<<grid, kHeadThreads, smem, stream>>>(p); break;
        case 2: head_param_grad_kernel<T, CO, 2><<<grid, kHeadThreads, smem, stream>>>(p); break;
        case 3: head_param_grad_kernel<T, CO, 3><<<grid, kHeadThreads, smem, stream>>>(p); break;
        default: head_param_grad_kernel<T, CO, 4><<<grid, kHeadThreads, smem, stream>>>(p); break;
    }
    return check_launch("ctu_head_param_grad");
}

static int head_loss_setup(HeadParams& p, int flags, int cout, const void* tgt0, const void* tgt1, int target_u8, double* sums,
                           int softmax_for_dice, float ce_lambda, float dice_lambda, int& pairs, const char* what) {
    pairs = (flags & (CTU_HEAD_SP | CTU_HEAD_SP_SOFTMAX)) ? 2 : 1;
    CTU_REQUIRE(!target_u8 || pairs == 2 || cout == 2, "%s: uint8 mask targets need two classes", what);
    p.tgt_u8 = target_u8 ? 1 : 0;
    CTU_REQUIRE(tgt0 && (pairs == 1 || tgt1) && sums, "%s: missing target / sums", what);
    CTU_REQUIRE(ce_lambda != 0.f || dice_lambda != 0.f, "%s: both loss weights are zero", what);
    CTU_REQUIRE(pairs == 2 || cout >= 2 || ce_lambda == 0.f, "%s: CrossEntropy needs at least two classes", what);
    // head_load_targets2 reads two voxels per load (uchar2 / float2): a target view at an odd byte (uint8) or 4-mod-8 byte
    // (float) offset would fault inside the kernel
    const uintptr_t talign = target_u8 ? 2 : 8;
    CTU_REQUIRE(reinterpret_cast<uintptr_t>(tgt0) % talign == 0 && reinterpret_cast<uintptr_t>(tgt1) % talign == 0,
                "%s: %s targets must be %d-byte aligned", what, target_u8 ? "uint8" : "float32", (int)talign);
    p.tgt0 = reinterpret_cast<const float*>(tgt0); p.tgt1 = reinterpret_cast<const float*>(tgt1); p.lsums = sums;
    p.softmax_for_dice = softmax_for_dice; p.want_ce = ce_lambda != 0.f;
    p.g_ce = ce_lambda; p.g_dice = dice_lambda;
    return CTU_OK;
}


// ------------------------------------------------------------------------------------------------ head -> hard labels
// Inference epilogue: hard_segm_from_tensor (utilities.py:103-124: argmax over the channel axis as float32, first maximum
// wins) of every head output, computed in the head kernel itself (same arithmetic as head_fwd_kernel + argmax_kernel) and
// written either as [n][spatial] planes (origins == NULL) or scattered into full [D][H][W] label volumes at the patch
// origins of a sliding-window pass -- the fp32 [B,2,p,p,p] outputs, the separate argmax pass and the stitch copies vanish.
template <typename T, int CO, int CBT>
__global__ void __launch_bounds__(kHeadThreads) head_labels_kernel(HeadParams p, const int* __restrict__ origins, int patch, int vd,
                                                                   int vh, int vw) {
    extern __shared__ float hsm[];
    float* wsm = hsm;
    float* bsm = hsm + CO * CBT * 8;
    load_head_weights<CO>(p, wsm, bsm);
    __syncthreads();
    const long long total = (long long)p.n * p.spatial;
    const bool sp = (p.flags & (CTU_HEAD_SP | CTU_HEAD_SP_SOFTMAX)) != 0;
    for (long long i = (long long)blockIdx.x * kHeadThreads + threadIdx.x; i < total; i += (long long)gridDim.x * kHeadThreads) {
        const int n = (int)(i / p.spatial);
        const long long s = i % p.spatial;
        HeadVals<CO> h;
        V8 xs[CBT];
        head_logits<T, CO, CBT>(p, wsm, bsm, n, s, h, xs);
        head_forward_chain<CO>(h, p.flags);
        float l0, l1 = 0.f;
        if (sp) {
            l0 = (h.o0[1] > h.o0[0] || (h.o0[1] != h.o0[1] && h.o0[0] == h.o0[0])) ? 1.f : 0.f;
            l1 = (h.o1[1] > h.o1[0] || (h.o1[1] != h.o1[1] && h.o1[0] == h.o1[0])) ? 1.f : 0.f;
        } else {
            int bi = 0;
            float best = h.sg[0];
#pragma unroll
            for (int c = 1; c < CO; ++c)
                if (h.sg[c] > best || (h.sg[c] != h.sg[c] && best == best)) best = h.sg[c], bi = c;
            l0 = (float)bi;
        }
        long long dst = i;
        if (origins != nullptr) {
            const int x = (int)(s % patch), y = (int)((s / patch) % patch), z = (int)(s / ((long long)patch * patch));
            dst = ((long long)(origins[3 * n] + z) * vh + origins[3 * n + 1] + y) * vw + origins[3 * n + 2] + x;
        }
        p.out0[dst] = l0;
        if (sp) p.out1[dst] = l1;
    }
}

template <typename T, int CO>
static int head_labels_launch(const HeadParams& p, const int* origins, int patch, int vd, int vh, int vw, cudaStream_t stream) {
    const size_t smem = (size_t)(CO * p.m.cb_total * 8 + 8) * sizeof(float);
    const long long total = (long long)p.n * p.spatial;
    const int grid = (int)((total + kHeadThreads - 1) / kHeadThreads > 148 * 32 ? 148 * 32 : (total + kHeadThreads - 1) / kHeadThreads);
    switch (p.m.cb_total) {
        case 1: head_labels_kernel<T, CO, 1><<<grid, kHeadThreads, smem, stream>>>(p, origins, patch, vd, vh, vw); break;
        case 2: head_labels_kernel<T, CO, 2><<<grid, kHeadThreads, smem, stream>>>(p, origins, patch, vd, vh, vw); break;
        case 3: head_labels_kernel<T, CO, 3><<<grid, kHeadThreads, smem, stream>>>(p, origins, patch, vd, vh, vw); break;
        default: head_labels_kernel<T, CO, 4><<<grid, kHeadThreads, smem, stream>>>(p, origins, patch, vd, vh, vw); break;
    }
    return check_launch("ctu_head_labels");
}

// ------------------------------------------------------------------------------------------------ head -> blended sums
// Overlapping sliding-window inference (preprocess.sliding_window_predict, DESIGN.md section 7b).  Every window voxel
// inside the [vd][vh][vw] volume adds, for each head output channel v (the values ctu_head_fwd writes, all in [0, 2] for
// a head with softmax / sigmoid), llrint(w * v * 2^40) to acc[out][c][z][y][x], with the separable window weight
// w = wt[z] * wt[p + y] * wt[2p + x] (fp32).  Integer sums do not depend on the order of the additions: the blended
// result is bit-identical whatever the batch, the window order or the number of ranks.  The return values of the 64-bit
// atomics are unused, so they compile to reductions (RED.E.ADD.64).
constexpr float kAccScale = 1099511627776.f;      // 2^40

__device__ __forceinline__ void acc_add(long long* a, float v) {
    atomicAdd(reinterpret_cast<unsigned long long*>(a), (unsigned long long)__float2ll_rn(v * kAccScale));
}

template <typename T, int CO, int CBT>
__global__ void __launch_bounds__(kHeadThreads) head_accum_kernel(HeadParams p, const int* __restrict__ origins, int patch,
                                                                  int vd, int vh, int vw, const float* __restrict__ wt,
                                                                  long long* __restrict__ acc) {
    extern __shared__ float hsm[];
    float* wsm = hsm;
    float* bsm = hsm + CO * CBT * 8;
    load_head_weights<CO>(p, wsm, bsm);
    __syncthreads();
    const long long total = (long long)p.n * p.spatial;
    const long long plane = (long long)vd * vh * vw;
    const bool sp = (p.flags & (CTU_HEAD_SP | CTU_HEAD_SP_SOFTMAX)) != 0;
    for (long long i = (long long)blockIdx.x * kHeadThreads + threadIdx.x; i < total; i += (long long)gridDim.x * kHeadThreads) {
        const int n = (int)(i / p.spatial);
        const long long s = i % p.spatial;
        const int x = (int)(s % patch), y = (int)((s / patch) % patch), z = (int)(s / ((long long)patch * patch));
        const int gz = origins[3 * n] + z, gy = origins[3 * n + 1] + y, gx = origins[3 * n + 2] + x;
        if (gz < 0 || gz >= vd || gy < 0 || gy >= vh || gx < 0 || gx >= vw) continue;   // outputs past the volume: dropped
        HeadVals<CO> h;
        V8 xs[CBT];
        head_logits<T, CO, CBT>(p, wsm, bsm, n, s, h, xs);
        head_forward_chain<CO>(h, p.flags);
        const float w = __ldg(wt + z) * __ldg(wt + patch + y) * __ldg(wt + 2 * patch + x);
        long long* a = acc + ((long long)gz * vh + gy) * vw + gx;
        if (sp) {
            acc_add(a, w * h.o0[0]);
            acc_add(a + plane, w * h.o0[1]);
            acc_add(a + 2 * plane, w * h.o1[0]);
            acc_add(a + 3 * plane, w * h.o1[1]);
        } else {
#pragma unroll
            for (int c = 0; c < CO; ++c) acc_add(a + c * plane, w * h.sg[c]);
        }
    }
}

template <typename T, int CO>
static int head_accum_launch(const HeadParams& p, const int* origins, int patch, int vd, int vh, int vw, const float* wt,
                             long long* acc, cudaStream_t stream) {
    const size_t smem = (size_t)(CO * p.m.cb_total * 8 + 8) * sizeof(float);
    const long long total = (long long)p.n * p.spatial;
    const int grid = (int)((total + kHeadThreads - 1) / kHeadThreads > 148 * 32 ? 148 * 32 : (total + kHeadThreads - 1) / kHeadThreads);
    switch (p.m.cb_total) {
        case 1: head_accum_kernel<T, CO, 1><<<grid, kHeadThreads, smem, stream>>>(p, origins, patch, vd, vh, vw, wt, acc); break;
        case 2: head_accum_kernel<T, CO, 2><<<grid, kHeadThreads, smem, stream>>>(p, origins, patch, vd, vh, vw, wt, acc); break;
        case 3: head_accum_kernel<T, CO, 3><<<grid, kHeadThreads, smem, stream>>>(p, origins, patch, vd, vh, vw, wt, acc); break;
        default: head_accum_kernel<T, CO, 4><<<grid, kHeadThreads, smem, stream>>>(p, origins, patch, vd, vh, vw, wt, acc); break;
    }
    return check_launch("ctu_head_accumulate");
}

// Finalize of the blended sums: labels[o] = argmax over the C channels of acc[o] (first maximum wins; the per-voxel
// normaliser is a positive common factor, so the integer sums decide) and, when probs[o] is given, the blended values
// acc * 2^-40 / (nz[z] * ny[y] * nx[x]) from the float64 per-axis normaliser tables norm = [nz | ny | nx].
// One pass over the accumulators; VEC: four voxels per thread, 16-byte loads and stores (the plane size is a multiple
// of 4 and the buffers are 16-byte aligned).
template <int C, bool VEC>
__global__ void window_finalize_kernel(const long long* __restrict__ acc, int n_out, int vd, int vh, int vw,
                                       const double* __restrict__ norm, float* l0, float* l1, float* q0, float* q1) {
    const long long plane = (long long)vd * vh * vw;
    const long long nitem = VEC ? plane >> 2 : plane;
    constexpr int V = VEC ? 4 : 1;
    for (long long it = (long long)blockIdx.x * blockDim.x + threadIdx.x; it < nitem; it += (long long)gridDim.x * blockDim.x) {
        const long long v0 = it * V;
        double r[V];
        if (q0 != nullptr) {
#pragma unroll
            for (int k = 0; k < V; ++k) {
                const long long v = v0 + k;
                const int x = (int)(v % vw), y = (int)((v / vw) % vh), z = (int)(v / ((long long)vw * vh));
                r[k] = 0x1p-40 / (norm[z] * norm[vd + y] * norm[vd + vh + x]);
            }
        }
        for (int o = 0; o < n_out; ++o) {
            long long a[C][V];
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const long long* src = acc + ((long long)o * C + c) * plane + v0;
                if constexpr (VEC) {
                    const longlong2 u = __ldg(reinterpret_cast<const longlong2*>(src));
                    const longlong2 w = __ldg(reinterpret_cast<const longlong2*>(src) + 1);
                    a[c][0] = u.x; a[c][1] = u.y; a[c][2] = w.x; a[c][3] = w.y;
                } else {
                    a[c][0] = __ldg(src);
                }
            }
            float lab[V];
#pragma unroll
            for (int k = 0; k < V; ++k) {
                int bi = 0;
#pragma unroll
                for (int c = 1; c < C; ++c)
                    if (a[c][k] > a[bi][k]) bi = c;
                lab[k] = (float)bi;
            }
            float* lo = o == 0 ? l0 : l1;
            if constexpr (VEC) *reinterpret_cast<float4*>(lo + v0) = make_float4(lab[0], lab[1], lab[2], lab[3]);
            else lo[v0] = lab[0];
            float* qo = o == 0 ? q0 : q1;
            if (qo == nullptr) continue;
#pragma unroll
            for (int c = 0; c < C; ++c) {
                float f[V];
#pragma unroll
                for (int k = 0; k < V; ++k) f[k] = (float)((double)a[c][k] * r[k]);
                float* dst = qo + (long long)c * plane + v0;
                if constexpr (VEC) *reinterpret_cast<float4*>(dst) = make_float4(f[0], f[1], f[2], f[3]);
                else dst[0] = f[0];
            }
        }
    }
}

template <int C>
static int window_finalize_launch(const long long* acc, int n_out, int vd, int vh, int vw, const double* norm, float* l0,
                                  float* l1, float* q0, float* q1, cudaStream_t stream) {
    const long long plane = (long long)vd * vh * vw;
    bool vec = plane % 4 == 0;
    for (const void* ptr : {(const void*)acc, (const void*)l0, (const void*)l1, (const void*)q0, (const void*)q1})
        vec = vec && (reinterpret_cast<uintptr_t>(ptr) & 15u) == 0;
    const long long items = vec ? plane / 4 : plane;
    const int grid = (int)((items + 255) / 256 > 148 * 16 ? 148 * 16 : (items + 255) / 256);
    if (vec) window_finalize_kernel<C, true><<<grid, 256, 0, stream>>>(acc, n_out, vd, vh, vw, norm, l0, l1, q0, q1);
    else window_finalize_kernel<C, false><<<grid, 256, 0, stream>>>(acc, n_out, vd, vh, vw, norm, l0, l1, q0, q1);
    return check_launch("ctu_window_finalize");
}

}  // namespace ctu

using namespace ctu;

extern "C" {

int ctu_head_fwd(int dtype, const void* const* h_srcs, const int* h_src_channels, int nsrc, const float* w,
                 const float* bias, int cout, int flags, float* out0, float* out1, int n, long long spatial,
                 ctu_stream stream) {
    HeadParams p = {};
    int rc = head_setup(p, h_srcs, h_src_channels, nsrc, w, bias, cout, flags, n, spatial, "ctu_head_fwd");
    if (rc != CTU_OK) return rc;
    const bool sp = (flags & (CTU_HEAD_SP | CTU_HEAD_SP_SOFTMAX)) != 0;
    CTU_REQUIRE(out0 && (!sp || out1), "ctu_head_fwd: missing output");
    p.out0 = out0; p.out1 = out1;
    const size_t smem = (size_t)(cout * p.m.cb_total * 8 + 8) * sizeof(float);
    const long long total = (long long)n * spatial;
    // forward has no reduction: use the full grid
    const int grid = (int)((total + kHeadThreads - 1) / kHeadThreads > 148 * 32 ? 148 * 32 : (total + kHeadThreads - 1) / kHeadThreads);
    CTU_DISPATCH_DTYPE(dtype, {
        switch (cout) {
            case 1: return head_fwd_launch<T, 1>(p, grid, smem, (cudaStream_t)stream);
            case 2: return head_fwd_launch<T, 2>(p, grid, smem, (cudaStream_t)stream);
            case 3: return head_fwd_launch<T, 3>(p, grid, smem, (cudaStream_t)stream);
            default: return head_fwd_launch<T, 4>(p, grid, smem, (cudaStream_t)stream);
        }
    });
    return CTU_OK;
}

int ctu_head_bwd(int dtype, const void* const* h_srcs, const int* h_src_channels, int nsrc, const float* w,
                 const float* bias, int cout, int flags, const float* dout0, const float* dout1, const float* out0, const float* out1, void* const* h_dsrcs,
                 float* dw, float* db, int n, long long spatial, ctu_stream stream) {
    HeadParams p = {};
    int rc = head_setup(p, h_srcs, h_src_channels, nsrc, w, bias, cout, flags, n, spatial, "ctu_head_bwd");
    if (rc != CTU_OK) return rc;
    const bool sp = (flags & (CTU_HEAD_SP | CTU_HEAD_SP_SOFTMAX)) != 0;
    CTU_REQUIRE((dw != nullptr) == (db != nullptr) && (sp ? (dout0 || dout1) : dout0 != nullptr),
                "ctu_head_bwd: missing gradient buffers");
    bool any_dsrc = false;
    for (int i = 0; i < nsrc; ++i) {
        p.dsrc[i] = h_dsrcs ? h_dsrcs[i] : nullptr;
        any_dsrc = any_dsrc || p.dsrc[i] != nullptr;
    }
    CTU_REQUIRE(dw != nullptr || any_dsrc, "ctu_head_bwd: nothing to compute");
    const int part = dw == nullptr ? 1 : (any_dsrc ? 0 : 2);
    p.dout0 = dout0; p.dout1 = dout1; p.dw = dw; p.db = db;
    p.fo0 = out0; p.fo1 = out1;
    if (dw != nullptr) {
        cudaError_t e = cudaMemsetAsync(dw, 0, sizeof(float) * cout * p.m.c_total, (cudaStream_t)stream);
        if (e == cudaSuccess) e = cudaMemsetAsync(db, 0, sizeof(float) * cout, (cudaStream_t)stream);
        if (e != cudaSuccess) {
            set_error("ctu_head_bwd: memset: %s", cudaGetErrorString(e));
            return (int)e;
        }
    }
    CTU_DISPATCH_DTYPE(dtype, {
        switch (cout) {
            case 1: return head_bwd_launch<T, 1>(p, part, (cudaStream_t)stream);
            case 2: return head_bwd_launch<T, 2>(p, part, (cudaStream_t)stream);
            case 3: return head_bwd_launch<T, 3>(p, part, (cudaStream_t)stream);
            default: return head_bwd_launch<T, 4>(p, part, (cudaStream_t)stream);
        }
    });
    return CTU_OK;
}

int ctu_head_loss_fwd(int dtype, const void* const* h_srcs, const int* h_src_channels, int nsrc, const float* w,
                      const float* bias, int cout, int flags, const void* target0, const void* target1, int target_u8,
                      int softmax_for_dice, float ce_lambda, float dice_lambda, double* sums, float* comps, float* mirror,
                      int n, long long spatial, ctu_stream stream) {
    HeadParams p = {};
    int rc = head_setup(p, h_srcs, h_src_channels, nsrc, w, bias, cout, flags, n, spatial, "ctu_head_loss_fwd");
    if (rc != CTU_OK) return rc;
    int pairs = 1;
    rc = head_loss_setup(p, flags, cout, target0, target1, target_u8, sums, softmax_for_dice, ce_lambda, dice_lambda, pairs,
                         "ctu_head_loss_fwd");
    if (rc != CTU_OK) return rc;
    CTU_REQUIRE(comps != nullptr, "ctu_head_loss_fwd: comps is null");
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(sums, 0, sizeof(double) * 4 * pairs * n, st);
    if (e != cudaSuccess) {
        set_error("ctu_head_loss_fwd: memset: %s", cudaGetErrorString(e));
        return (int)e;
    }
    CTU_DISPATCH_DTYPE(dtype, {
        if (pairs == 2) rc = head_loss_fwd_launch<T, 3, 2>(p, st);
        else switch (cout) {
            case 1: rc = head_loss_fwd_launch<T, 1, 1>(p, st); break;
            case 2: rc = head_loss_fwd_launch<T, 2, 1>(p, st); break;
            case 3: rc = head_loss_fwd_launch<T, 3, 1>(p, st); break;
            default: rc = head_loss_fwd_launch<T, 4, 1>(p, st); break;
        }
    });
    if (rc != CTU_OK) return rc;
    head_loss_finalize_kernel<<<1, 1, 0, st>>>(sums, pairs, n, spatial, ce_lambda, dice_lambda, comps, mirror);
    return check_launch("head_loss_finalize_kernel");
}

int ctu_head_loss_bwd(int dtype, const void* const* h_srcs, const int* h_src_channels, int nsrc, const float* w,
                      const float* bias, int cout, int flags, const void* target0, const void* target1, int target_u8,
                      int softmax_for_dice, float ce_lambda, float dice_lambda, const double* sums, void* const* h_dsrcs,
                      float* dlogits, int n, long long spatial, ctu_stream stream) {
    HeadParams p = {};
    int rc = head_setup(p, h_srcs, h_src_channels, nsrc, w, bias, cout, flags, n, spatial, "ctu_head_loss_bwd");
    if (rc != CTU_OK) return rc;
    int pairs = 1;
    rc = head_loss_setup(p, flags, cout, target0, target1, target_u8, const_cast<double*>(sums), softmax_for_dice, ce_lambda,
                         dice_lambda, pairs, "ctu_head_loss_bwd");
    if (rc != CTU_OK) return rc;
    CTU_REQUIRE(h_dsrcs != nullptr && dlogits != nullptr, "ctu_head_loss_bwd: missing output buffers");
    CTU_REQUIRE(reinterpret_cast<uintptr_t>(dlogits) % 8 == 0, "ctu_head_loss_bwd: dlogits must be 8-byte aligned (float2 stores)");
    for (int i = 0; i < nsrc; ++i) p.dsrc[i] = h_dsrcs[i];
    p.out0 = dlogits;
    cudaStream_t st = (cudaStream_t)stream;
    CTU_DISPATCH_DTYPE(dtype, {
        if (pairs == 2) return head_loss_bwd_launch<T, 3, 2>(p, st);
        switch (cout) {
            case 1: return head_loss_bwd_launch<T, 1, 1>(p, st);
            case 2: return head_loss_bwd_launch<T, 2, 1>(p, st);
            case 3: return head_loss_bwd_launch<T, 3, 1>(p, st);
            default: return head_loss_bwd_launch<T, 4, 1>(p, st);
        }
    });
    return CTU_OK;
}

int ctu_head_param_grad(int dtype, const void* const* h_srcs, const int* h_src_channels, int nsrc, const float* dlogits,
                        int cout, float* dw, float* db, int n, long long spatial, ctu_stream stream) {
    HeadParams p = {};
    static const float dummy_w = 0.f;
    int rc = head_setup(p, h_srcs, h_src_channels, nsrc, &dummy_w, nullptr, cout, 0, n, spatial, "ctu_head_param_grad");
    if (rc != CTU_OK) return rc;
    CTU_REQUIRE(dlogits && dw && db, "ctu_head_param_grad: null pointer");
    p.dout0 = dlogits; p.dw = dw; p.db = db;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(dw, 0, sizeof(float) * cout * p.m.c_total, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(db, 0, sizeof(float) * cout, st);
    if (e != cudaSuccess) {
        set_error("ctu_head_param_grad: memset: %s", cudaGetErrorString(e));
        return (int)e;
    }
    CTU_DISPATCH_DTYPE(dtype, {
        switch (cout) {
            case 1: return head_param_grad_launch<T, 1>(p, st);
            case 2: return head_param_grad_launch<T, 2>(p, st);
            case 3: return head_param_grad_launch<T, 3>(p, st);
            default: return head_param_grad_launch<T, 4>(p, st);
        }
    });
    return CTU_OK;
}

int ctu_head_labels(int dtype, const void* const* h_srcs, const int* h_src_channels, int nsrc, const float* w, const float* bias,
                    int cout, int flags, const int* origins, int patch, int vd, int vh, int vw, float* labels0, float* labels1,
                    int n, long long spatial, ctu_stream stream) {
    HeadParams p = {};
    int rc = head_setup(p, h_srcs, h_src_channels, nsrc, w, bias, cout, flags, n, spatial, "ctu_head_labels");
    if (rc != CTU_OK) return rc;
    const bool sp = (flags & (CTU_HEAD_SP | CTU_HEAD_SP_SOFTMAX)) != 0;
    CTU_REQUIRE(labels0 && (!sp || labels1), "ctu_head_labels: missing output");
    CTU_REQUIRE(origins == nullptr || (patch > 0 && (long long)patch * patch * patch == spatial && vd >= patch && vh >= patch && vw >= patch),
                "ctu_head_labels: scatter mode needs spatial = patch^3 inside the volume");
    p.out0 = labels0; p.out1 = labels1;
    CTU_DISPATCH_DTYPE(dtype, {
        switch (cout) {
            case 1: return head_labels_launch<T, 1>(p, origins, patch, vd, vh, vw, (cudaStream_t)stream);
            case 2: return head_labels_launch<T, 2>(p, origins, patch, vd, vh, vw, (cudaStream_t)stream);
            case 3: return head_labels_launch<T, 3>(p, origins, patch, vd, vh, vw, (cudaStream_t)stream);
            default: return head_labels_launch<T, 4>(p, origins, patch, vd, vh, vw, (cudaStream_t)stream);
        }
    });
    return CTU_OK;
}

int ctu_head_accumulate(int dtype, const void* const* h_srcs, const int* h_src_channels, int nsrc, const float* w,
                        const float* bias, int cout, int flags, const int* origins, int patch, int vd, int vh, int vw,
                        const float* weights, long long* acc, int n, long long spatial, ctu_stream stream) {
    HeadParams p = {};
    int rc = head_setup(p, h_srcs, h_src_channels, nsrc, w, bias, cout, flags, n, spatial, "ctu_head_accumulate");
    if (rc != CTU_OK) return rc;
    CTU_REQUIRE(origins && weights && acc, "ctu_head_accumulate: missing origins / weights / accumulators");
    CTU_REQUIRE(patch > 0 && (long long)patch * patch * patch == spatial && vd > 0 && vh > 0 && vw > 0,
                "ctu_head_accumulate: needs spatial = patch^3 and a non-empty volume");
    CTU_REQUIRE(flags & (CTU_HEAD_SOFTMAX | CTU_HEAD_SIGMOID | CTU_HEAD_SP_SOFTMAX),
                "ctu_head_accumulate: the head outputs must be bounded (softmax or sigmoid) for the fixed-point sums");
    CTU_DISPATCH_DTYPE(dtype, {
        switch (cout) {
            case 1: return head_accum_launch<T, 1>(p, origins, patch, vd, vh, vw, weights, acc, (cudaStream_t)stream);
            case 2: return head_accum_launch<T, 2>(p, origins, patch, vd, vh, vw, weights, acc, (cudaStream_t)stream);
            case 3: return head_accum_launch<T, 3>(p, origins, patch, vd, vh, vw, weights, acc, (cudaStream_t)stream);
            default: return head_accum_launch<T, 4>(p, origins, patch, vd, vh, vw, weights, acc, (cudaStream_t)stream);
        }
    });
    return CTU_OK;
}

int ctu_window_finalize(const long long* acc, int n_out, int channels, int vd, int vh, int vw, const double* norm,
                        float* labels0, float* labels1, float* probs0, float* probs1, ctu_stream stream) {
    CTU_REQUIRE(acc && labels0 && vd > 0 && vh > 0 && vw > 0 && (n_out == 1 || (n_out == 2 && labels1)),
                "ctu_window_finalize: bad arguments (n_out 1 or 2, one label volume per output)");
    CTU_REQUIRE(channels >= 1 && channels <= 4, "ctu_window_finalize: channels must be 1..4");
    CTU_REQUIRE(!probs0 || (norm && (n_out == 1 || probs1)), "ctu_window_finalize: probabilities need the normaliser "
                "tables and one output per head output");
    const cudaStream_t st = (cudaStream_t)stream;
    switch (channels) {
        case 1: return window_finalize_launch<1>(acc, n_out, vd, vh, vw, norm, labels0, labels1, probs0, probs1, st);
        case 2: return window_finalize_launch<2>(acc, n_out, vd, vh, vw, norm, labels0, labels1, probs0, probs1, st);
        case 3: return window_finalize_launch<3>(acc, n_out, vd, vh, vw, norm, labels0, labels1, probs0, probs1, st);
        default: return window_finalize_launch<4>(acc, n_out, vd, vh, vw, norm, labels0, labels1, probs0, probs1, st);
    }
}

}  // extern "C"
