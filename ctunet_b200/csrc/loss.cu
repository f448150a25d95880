// Soft Dice + CrossEntropy on fp32 NCDHW prediction / one-hot target pairs, and channel argmax.
//   dice_loss.forward          ctunet/utilities.py:39-50
//   CE + softmax + weighting   ctunet/pytorch/ProblemHandler.py:59-91, 228-298
//   hard_segm_from_tensor      ctunet/utilities.py:103-124
// One pass computes, per sample, sum(p*t), sum(p*p), sum(t*t) and the CE sum (double accumulators in
// global memory, warp-shuffle reductions); a second tiny kernel forms the two scalars so the step
// stays free of host synchronisation.
#include "loss_math.cuh"

namespace ctu {

constexpr int kLossThreads = 256;

template <int C>
__global__ void __launch_bounds__(kLossThreads) dice_ce_fwd_kernel(const float* __restrict__ pred,
                                                                   const float* __restrict__ target, long long spatial,
                                                                   int softmax_for_dice, int want_ce,
                                                                   double* __restrict__ sums) {
    const int b = blockIdx.y;
    const float* pb = pred + (long long)b * C * spatial;
    const float* tb = target + (long long)b * C * spatial;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    // four consecutive voxels per thread and iteration (16-byte loads) when the planes allow it
    const int V = (spatial % 4 == 0) ? 4 : 1;
    const long long nvec = spatial / V;
    for (long long sv = (long long)blockIdx.x * kLossThreads + threadIdx.x; sv < nvec; sv += (long long)gridDim.x * kLossThreads) {
        float xs[C][4], ts[C][4];
        if (V == 4) {
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const float4 a = __ldg(reinterpret_cast<const float4*>(pb + c * spatial) + sv);
                const float4 b4 = __ldg(reinterpret_cast<const float4*>(tb + c * spatial) + sv);
                xs[c][0] = a.x; xs[c][1] = a.y; xs[c][2] = a.z; xs[c][3] = a.w;
                ts[c][0] = b4.x; ts[c][1] = b4.y; ts[c][2] = b4.z; ts[c][3] = b4.w;
            }
        } else {
#pragma unroll
            for (int c = 0; c < C; ++c) {
                xs[c][0] = __ldg(pb + c * spatial + sv);
                ts[c][0] = __ldg(tb + c * spatial + sv);
            }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
        if (j >= V) break;
        float x[C], t[C], p[C], lse = 0.f;
#pragma unroll
        for (int c = 0; c < C; ++c) {
            x[c] = xs[c][j];
            t[c] = ts[c][j];
        }
        if (softmax_for_dice || want_ce) softmax_c<C>(x, p, lse);
        if (want_ce) {
            const int k = first_argmax<C>(t);
            float xk = x[0];
#pragma unroll
            for (int c = 1; c < C; ++c) xk = (c == k) ? x[c] : xk;
            acc[3] += lse - xk;
        }
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const float q = softmax_for_dice ? p[c] : x[c];
            acc[0] = fmaf(q, t[c], acc[0]);
            acc[1] = fmaf(q, q, acc[1]);
            acc[2] = fmaf(t[c], t[c], acc[2]);
        }
        }
    }
    __shared__ float red[kLossThreads / 32][4];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        float v = warp_sum(acc[i]);
        if (lane == 0) red[warp][i] = v;
    }
    __syncthreads();
    if (threadIdx.x < 4) {
        double v = 0.0;
        for (int wq = 0; wq < kLossThreads / 32; ++wq) v += (double)red[wq][threadIdx.x];
        atomicAdd(sums + b * 4 + threadIdx.x, v);
    }
}

__global__ void dice_ce_finalize_kernel(const double* __restrict__ sums, int b, long long spatial, float* out) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    const double eps = 0.0000001;
    double dsum = 0.0, ce = 0.0;
    for (int i = 0; i < b; ++i) {
        dsum += (sums[i * 4 + 0] + eps) / (sums[i * 4 + 1] + sums[i * 4 + 2] + eps);
        ce += sums[i * 4 + 3];
    }
    out[0] = (float)(ce / ((double)b * (double)spatial));
    out[1] = (float)(1.0 - 2.0 * dsum / (double)b);
}

template <int C>
__global__ void __launch_bounds__(kLossThreads) dice_ce_bwd_kernel(const float* __restrict__ pred,
                                                                   const float* __restrict__ target, int nb,
                                                                   long long spatial, int softmax_for_dice, int want_ce,
                                                                   const double* __restrict__ sums,
                                                                   const float* __restrict__ g,
                                                                   float* __restrict__ dpred) {
    const int b = blockIdx.y;
    const float* pb = pred + (long long)b * C * spatial;
    const float* tb = target + (long long)b * C * spatial;
    float* db = dpred + (long long)b * C * spatial;
    const double eps = 0.0000001;
    const double N = sums[b * 4 + 0] + eps, D = sums[b * 4 + 1] + sums[b * 4 + 2] + eps;
    const float g_ce = g[0], g_dice = g[1];
    // d dice / d q_c = -(2/B) * (t_c * D - 2 q_c N) / D^2
    const float kt = (float)(-2.0 / nb / D) * g_dice;
    const float kq = (float)(4.0 / nb * N / (D * D)) * g_dice;
    const float kce = want_ce ? g_ce / ((float)nb * (float)spatial) : 0.f;
    const int V = (spatial % 4 == 0) ? 4 : 1;
    const long long nvec = spatial / V;
    for (long long sv = (long long)blockIdx.x * kLossThreads + threadIdx.x; sv < nvec; sv += (long long)gridDim.x * kLossThreads) {
        float xs[C][4], ts[C][4], gs[C][4];
        if (V == 4) {
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const float4 a = __ldg(reinterpret_cast<const float4*>(pb + c * spatial) + sv);
                const float4 b4 = __ldg(reinterpret_cast<const float4*>(tb + c * spatial) + sv);
                xs[c][0] = a.x; xs[c][1] = a.y; xs[c][2] = a.z; xs[c][3] = a.w;
                ts[c][0] = b4.x; ts[c][1] = b4.y; ts[c][2] = b4.z; ts[c][3] = b4.w;
            }
        } else {
#pragma unroll
            for (int c = 0; c < C; ++c) {
                xs[c][0] = __ldg(pb + c * spatial + sv);
                ts[c][0] = __ldg(tb + c * spatial + sv);
            }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
        if (j >= V) break;
        float x[C], t[C], p[C], lse, gq[C], gx[C];
#pragma unroll
        for (int c = 0; c < C; ++c) {
            x[c] = xs[c][j];
            t[c] = ts[c][j];
        }
        if (softmax_for_dice || want_ce) softmax_c<C>(x, p, lse);
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const float q = softmax_for_dice ? p[c] : x[c];
            gq[c] = kt * t[c] + kq * q;
        }
        if (softmax_for_dice) {
            float dot = 0.f;
#pragma unroll
            for (int c = 0; c < C; ++c) dot = fmaf(gq[c], p[c], dot);
#pragma unroll
            for (int c = 0; c < C; ++c) gx[c] = p[c] * (gq[c] - dot);
        } else {
#pragma unroll
            for (int c = 0; c < C; ++c) gx[c] = gq[c];
        }
        if (want_ce) {
            const int k = first_argmax<C>(t);
#pragma unroll
            for (int c = 0; c < C; ++c) gx[c] += kce * (p[c] - (c == k ? 1.f : 0.f));
        }
#pragma unroll
        for (int c = 0; c < C; ++c) gs[c][j] = gx[c];
        }
        if (V == 4) {
#pragma unroll
            for (int c = 0; c < C; ++c)
                reinterpret_cast<float4*>(db + c * spatial)[sv] = make_float4(gs[c][0], gs[c][1], gs[c][2], gs[c][3]);
        } else {
#pragma unroll
            for (int c = 0; c < C; ++c) db[c * spatial + sv] = gs[c][0];
        }
    }
}

__global__ void argmax_kernel(const float* __restrict__ x, float* __restrict__ out, int c, long long spatial,
                              long long total) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const long long b = i / spatial, s = i % spatial;
    const float* xb = x + b * c * spatial + s;
    float best = xb[0];
    int bi = 0;
    for (int k = 1; k < c; ++k) {
        const float v = xb[(long long)k * spatial];
        if (v > best || (v != v && best == best)) {   // first maximum wins; NaN is maximal (torch.argmax)
            best = v;
            bi = k;
        }
    }
    out[i] = (float)bi;
}

// spatial % 4 == 0 selects the float4 path of the kernels above: every plane then starts 16-byte aligned iff the base does
static bool vec4_aligned(long long spatial, const void* a, const void* b, const void* c = nullptr) {
    const auto mis = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) != 0; };
    return spatial % 4 != 0 || !(mis(a) || mis(b) || mis(c));
}

static int loss_grid(long long spatial) {
    long long g = (spatial + kLossThreads - 1) / kLossThreads;
    const long long cap = 148 * 4;
    return (int)(g < cap ? g : cap);
}

}  // namespace ctu

using namespace ctu;

extern "C" {

int ctu_dice_ce_fwd(const float* pred, const float* target, int b, int c, long long spatial, int softmax_for_dice,
                    int want_ce, double* sums, float* out, ctu_stream stream) {
    CTU_REQUIRE(pred && target && sums && out && b > 0 && c >= 1 && c <= 4 && spatial > 0,
                "ctu_dice_ce_fwd: bad arguments (1 <= c <= 4)");
    CTU_REQUIRE(vec4_aligned(spatial, pred, target), "ctu_dice_ce_fwd: pred and target must be 16-byte aligned (float4 loads)");
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(sums, 0, sizeof(double) * 4 * b, st);
    if (e != cudaSuccess) {
        set_error("ctu_dice_ce_fwd: memset: %s", cudaGetErrorString(e));
        return (int)e;
    }
    dim3 grid(loss_grid(spatial), b);
    switch (c) {
        case 1: dice_ce_fwd_kernel<1><<<grid, kLossThreads, 0, st>>>(pred, target, spatial, softmax_for_dice, want_ce, sums); break;
        case 2: dice_ce_fwd_kernel<2><<<grid, kLossThreads, 0, st>>>(pred, target, spatial, softmax_for_dice, want_ce, sums); break;
        case 3: dice_ce_fwd_kernel<3><<<grid, kLossThreads, 0, st>>>(pred, target, spatial, softmax_for_dice, want_ce, sums); break;
        default: dice_ce_fwd_kernel<4><<<grid, kLossThreads, 0, st>>>(pred, target, spatial, softmax_for_dice, want_ce, sums); break;
    }
    dice_ce_finalize_kernel<<<1, 32, 0, st>>>(sums, b, spatial, out);
    return check_launch("ctu_dice_ce_fwd");
}

int ctu_dice_ce_bwd(const float* pred, const float* target, int b, int c, long long spatial, int softmax_for_dice,
                    int want_ce, const double* sums, const float* g, float* dpred, ctu_stream stream) {
    CTU_REQUIRE(pred && target && sums && g && dpred && b > 0 && c >= 1 && c <= 4 && spatial > 0,
                "ctu_dice_ce_bwd: bad arguments (1 <= c <= 4)");
    CTU_REQUIRE(vec4_aligned(spatial, pred, target, dpred),
                "ctu_dice_ce_bwd: pred, target and dpred must be 16-byte aligned (float4 loads / stores)");
    cudaStream_t st = (cudaStream_t)stream;
    dim3 grid(loss_grid(spatial) * 4, b);
    switch (c) {
        case 1: dice_ce_bwd_kernel<1><<<grid, kLossThreads, 0, st>>>(pred, target, b, spatial, softmax_for_dice, want_ce, sums, g, dpred); break;
        case 2: dice_ce_bwd_kernel<2><<<grid, kLossThreads, 0, st>>>(pred, target, b, spatial, softmax_for_dice, want_ce, sums, g, dpred); break;
        case 3: dice_ce_bwd_kernel<3><<<grid, kLossThreads, 0, st>>>(pred, target, b, spatial, softmax_for_dice, want_ce, sums, g, dpred); break;
        default: dice_ce_bwd_kernel<4><<<grid, kLossThreads, 0, st>>>(pred, target, b, spatial, softmax_for_dice, want_ce, sums, g, dpred); break;
    }
    return check_launch("ctu_dice_ce_bwd");
}

int ctu_argmax_channels(const float* x, float* out, int b, int c, long long spatial, ctu_stream stream) {
    CTU_REQUIRE(x && out && b > 0 && c > 0 && spatial > 0, "ctu_argmax_channels: bad arguments");
    const long long total = (long long)b * spatial;
    argmax_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(x, out, c, spatial, total);
    return check_launch("ctu_argmax_channels");
}

}  // extern "C"
