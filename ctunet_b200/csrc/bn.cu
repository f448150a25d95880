// BatchNorm3d (+ ReLU, + MaxPool3d(2,2)) forward / backward on the blocked layout.
// Reference: nn.BatchNorm3d + nn.ReLU(True) at ctunet/pytorch/models.py:27-28,31-32,39-40,43-44,
// nn.MaxPool3d(2,2) at models.py:190-191,233 (indices discarded).  HBM-bound glue: every thread
// moves whole 16/32-byte channel groups, statistics are reduced with warp shuffles.
#include "common.cuh"
#include <stdlib.h>

namespace ctu {

constexpr int kBnThreads = 256;
constexpr int kStatVoxPerThread = 32;

// Block-level reduction of NV per-thread values followed by one double atomic per value.
template <int NV>
__device__ __forceinline__ void block_atomic_add(const float (&vals)[NV], double* dst, int stride, int cvalid) {
    __shared__ float red[kBnThreads / 32][NV];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        float s = warp_sum(vals[i]);
        if (lane == 0) red[warp][i] = s;
    }
    __syncthreads();
    if (threadIdx.x < NV) {
        double s = 0.0;
#pragma unroll
        for (int wq = 0; wq < kBnThreads / 32; ++wq) s += (double)red[wq][threadIdx.x];
        // value i -> channel (i % 8), quantity (i / 8)
        const int ch = threadIdx.x & 7, q = threadIdx.x >> 3;
        if (ch < cvalid) atomicAdd(dst + (long long)q * stride + ch, s);
    }
    __syncthreads();
}

// sums[0*cpad + ch] = sum, sums[1*cpad + ch] = sum of squares.  grid = (chunks, phases*cb, n): the tensor holds
// `phases` copies of the cb natural channel blocks (phase-major output of the fused up-sampling stage; 1 otherwise)
template <typename T>
__global__ void __launch_bounds__(kBnThreads) bn_stats_kernel(const T* __restrict__ y, double* __restrict__ sums, int c,
                                                              int cb, long long spatial) {
    const int b = blockIdx.y % cb, n = blockIdx.z;
    const T* base = y + ((long long)n * gridDim.y + blockIdx.y) * spatial * 8;
    float acc[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = 0.f;
    for (long long s0 = (long long)blockIdx.x * kBnThreads * kStatVoxPerThread; s0 < spatial;
         s0 += (long long)gridDim.x * kBnThreads * kStatVoxPerThread) {
#pragma unroll 4
        for (int it = 0; it < kStatVoxPerThread; ++it) {
            long long s = s0 + (long long)it * kBnThreads + threadIdx.x;
            if (s < spatial) {
                V8 v = Vec8<T>::load(base + s * 8);
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    acc[j] += v.v[j];
                    acc[8 + j] = fmaf(v.v[j], v.v[j], acc[8 + j]);
                }
            }
        }
    }
    const int cpad = cb * 8;
    int cvalid = c - b * 8;
    if (cvalid > 8) cvalid = 8;
    block_atomic_add<16>(acc, sums + b * 8, cpad, cvalid);
}

// One thread per channel.  ss = scale | shift | mean | invstd (each cpad floats).
__global__ void bn_finalize_kernel(const double* __restrict__ sums, double count, const float* __restrict__ gamma,
                                   const float* __restrict__ beta, float* running_mean, float* running_var,
                                   long long* nbt, float momentum, float eps, int c, int cpad, int training,
                                   int n_updates, float* __restrict__ ss) {
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= cpad) return;
    float scale = 0.f, shift = 0.f, meanf = 0.f, invstd = 0.f;
    if (ch < c) {
        double mean, var;
        if (training) {
            mean = sums[ch] / count;
            var = sums[cpad + ch] / count - mean * mean;
            if (var < 0.0) var = 0.0;
            if (running_mean != nullptr && running_var != nullptr) {
                const double unbiased = count > 1.0 ? var * count / (count - 1.0) : var;
                float rm = running_mean[ch], rv = running_var[ch];
                for (int u = 0; u < n_updates; ++u) {
                    rm = (1.f - momentum) * rm + momentum * (float)mean;
                    rv = (1.f - momentum) * rv + momentum * (float)unbiased;
                }
                running_mean[ch] = rm;
                running_var[ch] = rv;
            }
        } else {
            mean = (double)running_mean[ch];
            var = (double)running_var[ch];
        }
        invstd = (float)(1.0 / sqrt(var + (double)eps));
        meanf = (float)mean;
        scale = gamma[ch] * invstd;
        shift = beta[ch] - meanf * scale;
    }
    ss[ch] = scale;
    ss[cpad + ch] = shift;
    ss[2 * cpad + ch] = meanf;
    ss[3 * cpad + ch] = invstd;
    if (ch == 0 && training && nbt != nullptr) *nbt += n_updates;
}

__global__ void bn_running_update_kernel(const double* __restrict__ sums, double count, float* running_mean,
                                         float* running_var, long long* nbt, float momentum, int c, int cpad,
                                         int n_updates) {
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch < c) {
        double mean = sums[ch] / count;
        double var = sums[cpad + ch] / count - mean * mean;
        if (var < 0.0) var = 0.0;
        const double unbiased = count > 1.0 ? var * count / (count - 1.0) : var;
        float rm = running_mean[ch], rv = running_var[ch];
        for (int u = 0; u < n_updates; ++u) {
            rm = (1.f - momentum) * rm + momentum * (float)mean;
            rv = (1.f - momentum) * rv + momentum * (float)unbiased;
        }
        running_mean[ch] = rm;
        running_var[ch] = rv;
    }
    if (ch == 0 && nbt != nullptr) *nbt += n_updates;
}

template <typename T>
__device__ __forceinline__ V8 bn_relu_apply(const V8& y, const float (&sc)[8], const float (&sh)[8]) {
    V8 a;
#pragma unroll
    for (int j = 0; j < 8; ++j) a.v[j] = round_to<T>(fmaxf(fmaf(y.v[j], sc[j], sh[j]), 0.f));
    return a;
}

// Dropout3d after the ReLU (models.py:34,46): a = k * relu(scale*y + shift), k = the keep factor of the (sample, channel),
// rounded ONCE to the storage type.  The factor multiplies the ReLU output rather than being folded into scale / shift: the
// backward pass re-elects the pooling arg-max from the unscaled value, and k >= 0 commutes with the max, so the pooled
// output is MaxPool3d(Dropout3d(a)) as models.py:233 orders them.
template <typename T>
__device__ __forceinline__ V8 bn_relu_drop_apply(const V8& y, const float (&sc)[8], const float (&sh)[8], const float (&k)[8]) {
    V8 a;
#pragma unroll
    for (int j = 0; j < 8; ++j) a.v[j] = round_to<T>(k[j] * fmaxf(fmaf(y.v[j], sc[j], sh[j]), 0.f));
    return a;
}

// keep factors [n][cpad] of channel block b of sample n (DROP kernels only)
__device__ __forceinline__ void load_keep(const float* __restrict__ keep, int n, int b, int cpad, float (&k)[8]) {
#pragma unroll
    for (int j = 0; j < 8; ++j) k[j] = __ldg(keep + (long long)n * cpad + b * 8 + j);
}

constexpr int kVoxPerThread = 4;   // plain (unpooled) kernels: voxels per thread, strided by the block size

// a = relu(scale*y + shift); grid = (chunks, cb, n)
// Training-mode finalisation folded into the forward kernels (ctu_bn_relu_fwd_train): every block derives scale / shift of
// its 8 channels from the batch sums (what bn_finalize_kernel computes); the first block of each channel block also
// writes ss for the backward pass and moves the running statistics.  One launch less per BatchNorm on the critical path.
struct BnFin {
    const double* sums;      // nullptr: read ss (the separate ctu_bn_finalize path, e.g. eval mode)
    double count;
    const float* gamma;
    const float* beta;
    float* running_mean;
    float* running_var;
    long long* nbt;
    float momentum, eps;
    int c, n_updates;
    float* ss_out;
};

template <bool FOLD>
__device__ __forceinline__ void bn_scale_shift(const BnFin& f, const float* __restrict__ ss, int b, int cpad, bool writer,
                                               float (&sc)[8], float (&sh)[8]) {
    if constexpr (!FOLD) {     // (compile-time: the plain kernels stay exactly what they were before the fold existed)
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            sc[j] = __ldg(ss + b * 8 + j);
            sh[j] = __ldg(ss + cpad + b * 8 + j);
        }
        return;
    }
    __shared__ float s_sc[8], s_sh[8];
    if (threadIdx.x < 8) {
        const int ch = b * 8 + threadIdx.x;
        float scale = 0.f, shift = 0.f, meanf = 0.f, invstd = 0.f;
        if (ch < f.c) {
            const double mean = f.sums[ch] / f.count;
            double var = f.sums[cpad + ch] / f.count - mean * mean;
            if (var < 0.0) var = 0.0;
            if (writer && f.running_mean != nullptr && f.running_var != nullptr) {
                const double unbiased = f.count > 1.0 ? var * f.count / (f.count - 1.0) : var;
                float rm = f.running_mean[ch], rv = f.running_var[ch];
                for (int u = 0; u < f.n_updates; ++u) {
                    rm = (1.f - f.momentum) * rm + f.momentum * (float)mean;
                    rv = (1.f - f.momentum) * rv + f.momentum * (float)unbiased;
                }
                f.running_mean[ch] = rm;
                f.running_var[ch] = rv;
            }
            invstd = (float)(1.0 / sqrt(var + (double)f.eps));
            meanf = (float)mean;
            scale = f.gamma[ch] * invstd;
            shift = f.beta[ch] - meanf * scale;
        }
        s_sc[threadIdx.x] = scale;
        s_sh[threadIdx.x] = shift;
        if (writer) {
            f.ss_out[ch] = scale;
            f.ss_out[cpad + ch] = shift;
            f.ss_out[2 * cpad + ch] = meanf;
            f.ss_out[3 * cpad + ch] = invstd;
            if (ch == 0 && f.nbt != nullptr) *f.nbt += f.n_updates;
        }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        sc[j] = s_sc[j];
        sh[j] = s_sh[j];
    }
}

template <typename T, bool FOLD, bool DROP>
__global__ void __launch_bounds__(kBnThreads) bn_relu_fwd_kernel(const T* __restrict__ y, const float* __restrict__ ss,
                                                                 T* __restrict__ a, int cb, long long spatial, BnFin fin,
                                                                 const float* __restrict__ keep) {
    const int b = blockIdx.y, n = blockIdx.z;
    const int cpad = cb * 8;
    float sc[8], sh[8], kf[8];
    bn_scale_shift<FOLD>(fin, ss, b, cpad, blockIdx.x == 0 && n == 0, sc, sh);
    if constexpr (DROP) load_keep(keep, n, b, cpad, kf);
    const long long base = ((long long)n * cb + b) * spatial;
    const long long s0 = (long long)blockIdx.x * kBnThreads * kVoxPerThread + threadIdx.x;
    V8 v[kVoxPerThread];
#pragma unroll
    for (int it = 0; it < kVoxPerThread; ++it) {
        const long long s = s0 + (long long)it * kBnThreads;
        if (s < spatial) v[it] = Vec8<T>::load(y + (base + s) * 8);
    }
#pragma unroll
    for (int it = 0; it < kVoxPerThread; ++it) {
        const long long s = s0 + (long long)it * kBnThreads;
        if (s < spatial) {
            if constexpr (DROP) Vec8<T>::store(a + (base + s) * 8, bn_relu_drop_apply<T>(v[it], sc, sh, kf));
            else Vec8<T>::store(a + (base + s) * 8, bn_relu_apply<T>(v[it], sc, sh));
        }
    }
}

// One thread per LOW-resolution voxel and its 8 children (d, h, w even).
//   POOL:  y, a natural [n][cb][d][h][w][8]; pooled = maxpool 2x2x2 of a.
//   S2D:   y phase-major [n][8*cb][d/2][h/2][w/2][8] (output of the fused up-sampling stage, block = q*cb + b,
//          q = qd*4 + qh*2 + qw), a natural.
//   DROP:  a (and pooled) carry the Dropout3d keep factors (natural input only).
template <typename T, bool S2D, bool FOLD, bool DROP>
__global__ void __launch_bounds__(kBnThreads) bn_relu_child_fwd_kernel(const T* __restrict__ y,
                                                                       const float* __restrict__ ss, T* __restrict__ a,
                                                                       T* __restrict__ pooled, int cb, int d, int h,
                                                                       int w, BnFin fin, const float* __restrict__ keep) {
    static_assert(!(S2D && DROP), "a phase-major BatchNorm input never precedes a dropout site");
    const int b = blockIdx.y, n = blockIdx.z;
    const int cpad = cb * 8;
    float sc[8], sh[8], kf[8];
    bn_scale_shift<FOLD>(fin, ss, b, cpad, blockIdx.x == 0 && n == 0, sc, sh);
    if constexpr (DROP) load_keep(keep, n, b, cpad, kf);
    const int pd = d / 2, ph = h / 2, pw = w / 2;
    const long long pspatial = (long long)pd * ph * pw;
    const long long ps = (long long)blockIdx.x * kBnThreads + threadIdx.x;
    if (ps >= pspatial) return;
    const int px = (int)(ps % pw);
    const int py = (int)((ps / pw) % ph);
    const int pz = (int)(ps / ((long long)pw * ph));
    const long long spatial = (long long)d * h * w;
    const long long base = ((long long)n * cb + b) * spatial;
    V8 mx;
#pragma unroll
    for (int j = 0; j < 8; ++j) mx.v[j] = 0.f;   // a >= 0 after ReLU
    V8 in[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const int z = 2 * pz + (q >> 2), yy = 2 * py + ((q >> 1) & 1), x = 2 * px + (q & 1);
        const long long off = S2D ? ((((long long)n * 8 + q) * cb + b) * pspatial + ps) * 8
                                  : (base + ((long long)z * h + yy) * w + x) * 8;
        in[q] = Vec8<T>::load(y + off);
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const int z = 2 * pz + (q >> 2), yy = 2 * py + ((q >> 1) & 1), x = 2 * px + (q & 1);
        V8 r;
        if constexpr (DROP) r = bn_relu_drop_apply<T>(in[q], sc, sh, kf);
        else r = bn_relu_apply<T>(in[q], sc, sh);
        Vec8<T>::store(a + (base + ((long long)z * h + yy) * w + x) * 8, r);
        if (!S2D) {
#pragma unroll
            for (int j = 0; j < 8; ++j) mx.v[j] = fmaxf(mx.v[j], r.v[j]);
        }
    }
    if (!S2D) Vec8<T>::store(pooled + (((long long)n * cb + b) * pspatial + ps) * 8, mx);
}

// ---------------------------------------------------------------------------- backward
// Gradient entering the BatchNorm output: dz = (dA + [child is the first max of its window] * dP) * [a > 0].
// DROP: dz = k * (dA + [winner] * dP) * [scale*y + shift > 0] with the keep factors of the forward (the batch statistics
// stay those of y: BatchNorm comes before the dropout).
// MODE 0: one voxel at a time (kVoxPerThread per thread); MODE 1 (pool): the 8 children of one pooled voxel;
// MODE 2 (s2d): the 8 children of one low-res voxel with y / dy phase-major and dA natural.
struct BwdArgs {
    const void* y;
    const float* ss;
    const float* gamma;
    const void* dA;
    const void* dP;
    double* sums2;        // reduce: output; apply: input
    const float* keep;    // Dropout3d keep factors [n][cpad] (DROP kernels)
    double count;
    void* dy;
    float* dgamma;
    float* dbeta;
    int c, cb, d, h, w;
    long long nblk;       // chunks of kBnThreads (x kVoxPerThread in mode 0) voxels per (n, block) plane
};

template <typename T, int MODE, bool APPLY, bool DROP>
__global__ void __launch_bounds__(kBnThreads, 2) bn_relu_bwd_kernel(BwdArgs p) {
    constexpr bool POOL = MODE == 1, S2D = MODE == 2;     // MODE 3: the child structure on a natural, unpooled tensor
    static_assert(!(S2D && DROP), "a phase-major BatchNorm input never precedes a dropout site");
    const int b = blockIdx.y, n = blockIdx.z;
    const int cpad = p.cb * 8;
    __shared__ float kk[16];
    if (APPLY) {
        if (threadIdx.x < 16) {
            const int j = threadIdx.x & 7, q = threadIdx.x >> 3;
            kk[threadIdx.x] = (float)(p.sums2[q * cpad + b * 8 + j] / p.count);   // mean(dz) | mean(dz * xhat)
            if (blockIdx.x == 0 && n == 0 && b * 8 + j < p.c) {
                if (q == 0) p.dbeta[b * 8 + j] = (float)p.sums2[b * 8 + j];
                else p.dgamma[b * 8 + j] = (float)p.sums2[cpad + b * 8 + j];
            }
        }
        __syncthreads();
    }
    float sc[8], sh[8], mean[8], invstd[8], k1[8], k2[8], kf[8];
    if constexpr (DROP) load_keep(p.keep, n, b, cpad, kf);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        sc[j] = __ldg(p.ss + b * 8 + j);
        sh[j] = __ldg(p.ss + cpad + b * 8 + j);
        mean[j] = __ldg(p.ss + 2 * cpad + b * 8 + j);
        invstd[j] = __ldg(p.ss + 3 * cpad + b * 8 + j);
        if (APPLY) {
            k1[j] = kk[j];
            k2[j] = kk[8 + j];
        }
    }
    const T* y = reinterpret_cast<const T*>(p.y);
    const T* dA = reinterpret_cast<const T*>(p.dA);
    const T* dP = reinterpret_cast<const T*>(p.dP);
    T* dy = reinterpret_cast<T*>(p.dy);
    const long long spatial = (long long)p.d * p.h * p.w;
    const long long base = ((long long)n * p.cb + b) * spatial;
    float acc[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = 0.f;

    // (the reduce pass walks several chunks per block: its 16 double atomics per block all hit the same
    // addresses and serialise at ~1 ns each, so fewer, fatter blocks)
    for (long long blk = blockIdx.x; blk < p.nblk; blk += gridDim.x) {
    if (MODE == 0) {
        const long long s0 = blk * kBnThreads * kVoxPerThread + threadIdx.x;
        V8 yv[kVoxPerThread], g[kVoxPerThread];
#pragma unroll
        for (int it = 0; it < kVoxPerThread; ++it) {
            const long long s = s0 + (long long)it * kBnThreads;
            if (s < spatial) {
                yv[it] = Vec8<T>::load(y + (base + s) * 8);
                g[it] = Vec8<T>::load(dA + (base + s) * 8);
            }
        }
#pragma unroll
        for (int it = 0; it < kVoxPerThread; ++it) {
            const long long s = s0 + (long long)it * kBnThreads;
            if (s < spatial) {
                V8 o;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float av = fmaf(yv[it].v[j], sc[j], sh[j]);
                    const float dz = av > 0.f ? (DROP ? kf[j] * g[it].v[j] : g[it].v[j]) : 0.f;
                    const float xhat = (yv[it].v[j] - mean[j]) * invstd[j];
                    if (APPLY) {
                        o.v[j] = sc[j] * (dz - k1[j] - xhat * k2[j]);
                    } else {
                        acc[j] += dz;
                        acc[8 + j] = fmaf(dz, xhat, acc[8 + j]);
                    }
                }
                if (APPLY) Vec8<T>::store(dy + (base + s) * 8, o);
            }
        }
    } else {
        const int pd = p.d / 2, ph = p.h / 2, pw = p.w / 2;
        const long long pspatial = (long long)pd * ph * pw;
        const long long ps = blk * kBnThreads + threadIdx.x;
        if (ps < pspatial) {
            const int px = (int)(ps % pw);
            const int py = (int)((ps / pw) % ph);
            const int pz = (int)(ps / ((long long)pw * ph));
            long long offa[8], offy[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int z = 2 * pz + (q >> 2), yy = 2 * py + ((q >> 1) & 1), x = 2 * px + (q & 1);
                offa[q] = (base + ((long long)z * p.h + yy) * p.w + x) * 8;
                offy[q] = S2D ? ((((long long)n * 8 + q) * p.cb + b) * pspatial + ps) * 8 : offa[q];
            }
            V8 gp;
            if (POOL) gp = Vec8<T>::load(dP + (((long long)n * p.cb + b) * pspatial + ps) * 8);
            // av: the activation BEFORE rounding to the storage type.  Rounding is monotone, so the maximum of
            // the rounded values is the rounded maximum (forward/backward stay consistent) while values that
            // collide in bf16 still elect the arg-max an fp32 evaluation would.  The children stay in their storage
            // form (Raw8) and av is recomputed on use: the pooled variant fits 128 registers without spilling.
            // bf16: the two x-neighbours of a cell are 32 contiguous bytes -> one 256-bit access for the pair (half the
            // load / store instructions and fully used sectors); the phase-major tensor (S2D: y, dy) has no such pairs
            constexpr bool PAIR = sizeof(T) == 2 && !POOL && APPLY;   // (measured: apply 102 -> 94 us, but the reduce pass 72 -> 82 us; the pooled variant is at its register limit)
            Raw8<T> yr[8];
            if constexpr (PAIR && !S2D) {
#pragma unroll
                for (int q = 0; q < 8; q += 2)
                    ldg256(y + offy[q], reinterpret_cast<Raw8<__nv_bfloat16>&>(yr[q]).u, reinterpret_cast<Raw8<__nv_bfloat16>&>(yr[q + 1]).u);
            } else {
#pragma unroll
                for (int q = 0; q < 8; ++q) yr[q].load(y + offy[q]);
            }
            int win[8];
            if (POOL) {
                // first maximum in (d, h, w) scan order, strict '>' like torch's max_pool3d
                float best[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const V8 yq = yr[q].get();
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float a = fmaxf(fmaf(yq.v[j], sc[j], sh[j]), 0.f);
                        if (q == 0 || a > best[j]) {
                            best[j] = a;
                            win[j] = q;
                        }
                    }
                }
            }
            uint4 gpair = make_uint4(0, 0, 0, 0), opair = make_uint4(0, 0, 0, 0);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                V8 g;
                if (dA != nullptr) {
                    if constexpr (PAIR) {
                        if ((q & 1) == 0) {
                            uint4 g0;
                            ldg256(dA + offa[q], g0, gpair);
                            g = unpack_bf16x8(g0);
                        } else {
                            g = unpack_bf16x8(gpair);
                        }
                    } else {
                        g = Vec8<T>::load(dA + offa[q]);
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 8; ++j) g.v[j] = 0.f;
                }
                const V8 yq = yr[q].get();
                V8 o;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    float dz = g.v[j];
                    if (POOL) dz += (win[j] == q) ? gp.v[j] : 0.f;
                    if constexpr (DROP) dz *= kf[j];
                    dz = fmaf(yq.v[j], sc[j], sh[j]) > 0.f ? dz : 0.f;
                    const float xhat = (yq.v[j] - mean[j]) * invstd[j];
                    if (APPLY) {
                        o.v[j] = sc[j] * (dz - k1[j] - xhat * k2[j]);
                    } else {
                        acc[j] += dz;
                        acc[8 + j] = fmaf(dz, xhat, acc[8 + j]);
                    }
                }
                if (APPLY) {
                    if constexpr (PAIR && !S2D) {
                        if ((q & 1) == 0) opair = pack_bf16x8(o);
                        else stg256(dy + offy[q - 1], opair, pack_bf16x8(o));
                    } else {
                        Vec8<T>::store(dy + offy[q], o);
                    }
                }
            }
        }
    }
    }
    if (!APPLY) {
        int cvalid = p.c - b * 8;
        if (cvalid > 8) cvalid = 8;
        block_atomic_add<16>(acc, p.sums2 + b * 8, cpad, cvalid);
    }
}

}  // namespace ctu

using namespace ctu;

extern "C" {

int ctu_bn_stats(int dtype, const void* y, int c, int phases, int n, long long spatial, double* sums, ctu_stream stream) {
    const bool prezeroed = (phases & CTU_ACCUM_PREZEROED) != 0;
    phases &= ~CTU_ACCUM_PREZEROED;
    CTU_REQUIRE(y && sums && c > 0 && phases > 0 && n > 0 && spatial > 0, "ctu_bn_stats: bad arguments");
    const int cb = (c + 7) / 8;
    cudaError_t e = prezeroed ? cudaSuccess : cudaMemsetAsync(sums, 0, sizeof(double) * 2 * cb * 8, (cudaStream_t)stream);
    if (e != cudaSuccess) {
        set_error("ctu_bn_stats: memset: %s", cudaGetErrorString(e));
        return (int)e;
    }
    long long gx = cdiv(spatial, (long long)kBnThreads * kStatVoxPerThread);
    dim3 grid((unsigned)gx, phases * cb, n);
    CTU_DISPATCH_DTYPE(dtype, (bn_stats_kernel<T><<<grid, kBnThreads, 0, (cudaStream_t)stream>>>((const T*)y, sums, c, cb, spatial)));
    return check_launch("ctu_bn_stats");
}

int ctu_bn_finalize(const double* sums, double count, const float* gamma, const float* beta, float* running_mean,
                    float* running_var, long long* num_batches_tracked, float momentum, float eps, int c,
                    int training, int n_updates, float* ss, ctu_stream stream) {
    CTU_REQUIRE(gamma && beta && ss && c > 0, "ctu_bn_finalize: bad arguments");
    CTU_REQUIRE(training ? (sums != nullptr && count > 0) : (running_mean && running_var), "ctu_bn_finalize: missing statistics");
    const int cpad = (c + 7) / 8 * 8;
    bn_finalize_kernel<<<cdiv(cpad, 128), 128, 0, (cudaStream_t)stream>>>(sums, count, gamma, beta, running_mean, running_var, num_batches_tracked, momentum, eps, c, cpad, training, n_updates, ss);
    return check_launch("ctu_bn_finalize");
}

int ctu_bn_running_update(const double* sums, double count, float* running_mean, float* running_var,
                          long long* num_batches_tracked, float momentum, int c, int n_updates, ctu_stream stream) {
    CTU_REQUIRE(sums && running_mean && running_var && c > 0 && count > 0, "ctu_bn_running_update: bad arguments");
    const int cpad = (c + 7) / 8 * 8;
    bn_running_update_kernel<<<cdiv(cpad, 128), 128, 0, (cudaStream_t)stream>>>(sums, count, running_mean, running_var, num_batches_tracked, momentum, c, cpad, n_updates);
    return check_launch("ctu_bn_running_update");
}

static int bn_relu_fwd_launch(int dtype, const void* y, const float* ss, void* a, void* pooled, int c, int n, int d, int h,
                              int w, int y_phase_major, const BnFin& fin, const float* keep, ctu_stream stream,
                              const char* what) {
    CTU_REQUIRE(y && (ss || fin.sums) && a && c > 0 && n > 0 && d > 0 && h > 0 && w > 0, "%s: bad arguments", what);
    CTU_REQUIRE(!(y_phase_major && pooled), "%s: a phase-major input is never pooled", what);
    CTU_REQUIRE(!(y_phase_major && keep), "%s: a phase-major input never carries dropout keep factors", what);
    const bool drop = keep != nullptr;
    const int cb = (c + 7) / 8;
    const long long spatial = (long long)d * h * w;
    const bool fold = fin.sums != nullptr;
    cudaStream_t st = (cudaStream_t)stream;
    if (pooled != nullptr || y_phase_major) {
        CTU_REQUIRE(d % 2 == 0 && h % 2 == 0 && w % 2 == 0, "%s: needs even dims (%d,%d,%d)", what, d, h, w);
        dim3 grid(cdiv(spatial / 8, kBnThreads), cb, n);
        CTU_DISPATCH_DTYPE(dtype, {
            if (y_phase_major && fold) bn_relu_child_fwd_kernel<T, true, true, false><<<grid, kBnThreads, 0, st>>>((const T*)y, ss, (T*)a, nullptr, cb, d, h, w, fin, nullptr);
            else if (y_phase_major) bn_relu_child_fwd_kernel<T, true, false, false><<<grid, kBnThreads, 0, st>>>((const T*)y, ss, (T*)a, nullptr, cb, d, h, w, fin, nullptr);
            else if (fold && drop) bn_relu_child_fwd_kernel<T, false, true, true><<<grid, kBnThreads, 0, st>>>((const T*)y, ss, (T*)a, (T*)pooled, cb, d, h, w, fin, keep);
            else if (drop) bn_relu_child_fwd_kernel<T, false, false, true><<<grid, kBnThreads, 0, st>>>((const T*)y, ss, (T*)a, (T*)pooled, cb, d, h, w, fin, keep);
            else if (fold) bn_relu_child_fwd_kernel<T, false, true, false><<<grid, kBnThreads, 0, st>>>((const T*)y, ss, (T*)a, (T*)pooled, cb, d, h, w, fin, nullptr);
            else bn_relu_child_fwd_kernel<T, false, false, false><<<grid, kBnThreads, 0, st>>>((const T*)y, ss, (T*)a, (T*)pooled, cb, d, h, w, fin, nullptr);
        });
    } else {
        dim3 grid(cdiv(spatial, kBnThreads * kVoxPerThread), cb, n);
        CTU_DISPATCH_DTYPE(dtype, {
            if (fold && drop) bn_relu_fwd_kernel<T, true, true><<<grid, kBnThreads, 0, st>>>((const T*)y, ss, (T*)a, cb, spatial, fin, keep);
            else if (drop) bn_relu_fwd_kernel<T, false, true><<<grid, kBnThreads, 0, st>>>((const T*)y, ss, (T*)a, cb, spatial, fin, keep);
            else if (fold) bn_relu_fwd_kernel<T, true, false><<<grid, kBnThreads, 0, st>>>((const T*)y, ss, (T*)a, cb, spatial, fin, nullptr);
            else bn_relu_fwd_kernel<T, false, false><<<grid, kBnThreads, 0, st>>>((const T*)y, ss, (T*)a, cb, spatial, fin, nullptr);
        });
    }
    return check_launch(what);
}

int ctu_bn_relu_fwd_drop(int dtype, const void* y, const float* ss, void* a, void* pooled, int c, int n, int d, int h,
                         int w, int y_phase_major, const float* keep, ctu_stream stream) {
    BnFin fin = {};
    return bn_relu_fwd_launch(dtype, y, ss, a, pooled, c, n, d, h, w, y_phase_major, fin, keep, stream,
                              keep ? "ctu_bn_relu_fwd_drop" : "ctu_bn_relu_fwd");
}

int ctu_bn_relu_fwd(int dtype, const void* y, const float* ss, void* a, void* pooled, int c, int n, int d, int h, int w,
                    int y_phase_major, ctu_stream stream) {
    return ctu_bn_relu_fwd_drop(dtype, y, ss, a, pooled, c, n, d, h, w, y_phase_major, nullptr, stream);
}

int ctu_bn_relu_fwd_train_drop(int dtype, const void* y, const double* sums, double count, const float* gamma,
                               const float* beta, float* running_mean, float* running_var, long long* num_batches_tracked,
                               float momentum, float eps, int n_updates, float* ss, void* a, void* pooled, int c, int n,
                               int d, int h, int w, int y_phase_major, const float* keep, ctu_stream stream) {
    const char* what = keep ? "ctu_bn_relu_fwd_train_drop" : "ctu_bn_relu_fwd_train";
    CTU_REQUIRE(sums && gamma && beta && ss && count > 0, "%s: bad arguments", what);
    BnFin fin = {sums, count, gamma, beta, running_mean, running_var, num_batches_tracked, momentum, eps, c, n_updates, ss};
    return bn_relu_fwd_launch(dtype, y, ss, a, pooled, c, n, d, h, w, y_phase_major, fin, keep, stream, what);
}

int ctu_bn_relu_fwd_train(int dtype, const void* y, const double* sums, double count, const float* gamma, const float* beta,
                          float* running_mean, float* running_var, long long* num_batches_tracked, float momentum, float eps,
                          int n_updates, float* ss, void* a, void* pooled, int c, int n, int d, int h, int w,
                          int y_phase_major, ctu_stream stream) {
    return ctu_bn_relu_fwd_train_drop(dtype, y, sums, count, gamma, beta, running_mean, running_var, num_batches_tracked,
                                      momentum, eps, n_updates, ss, a, pooled, c, n, d, h, w, y_phase_major, nullptr, stream);
}

static int bn_bwd(int dtype, BwdArgs& p, int n, bool apply, int y_phase_major, cudaStream_t stream, const char* what) {
    const long long spatial = (long long)p.d * p.h * p.w;
    const bool pool = p.dP != nullptr;
    if ((pool || y_phase_major) && (p.d % 2 || p.h % 2 || p.w % 2)) {
        set_error("%s: needs even dims", what);
        return CTU_ERR_INVALID;
    }
    if (pool && y_phase_major) {
        set_error("%s: a phase-major BatchNorm input is never pooled", what);
        return CTU_ERR_INVALID;
    }
    if (!pool && p.dA == nullptr) {
        set_error("%s: missing gradient", what);
        return CTU_ERR_INVALID;
    }
    if (y_phase_major && p.keep) {
        set_error("%s: a phase-major BatchNorm input never carries dropout keep factors", what);
        return CTU_ERR_INVALID;
    }
    const bool drop = p.keep != nullptr;
    // unpooled natural tensors with even dims also take the 8-children-per-thread structure (mode 3): measured 2x
    // faster than the strided one-voxel-at-a-time loop of mode 0
    const bool even = !(p.d % 2 || p.h % 2 || p.w % 2);
    const int mode = pool ? 1 : (y_phase_major ? 2 : (even ? 3 : 0));
    p.nblk = mode ? cdiv(spatial / 8, kBnThreads) : cdiv(spatial, kBnThreads * kVoxPerThread);
    long long gx = p.nblk;
    if (!apply) {      // reduce pass: a few fat blocks per SM (every block ends with 16 same-address double atomics)
        static const long long cap = getenv("CTU_BN_CAP") ? atoll(getenv("CTU_BN_CAP")) : 148 * 4;
        const long long want = (cap + (long long)p.cb * n - 1) / ((long long)p.cb * n);
        if (gx > want) gx = want;
    }
    dim3 grid((unsigned)gx, p.cb, n);
    CTU_DISPATCH_DTYPE(dtype, {
        if (drop) {
            if (mode == 1 && apply) bn_relu_bwd_kernel<T, 1, true, true><<<grid, kBnThreads, 0, stream>>>(p);
            else if (mode == 1) bn_relu_bwd_kernel<T, 1, false, true><<<grid, kBnThreads, 0, stream>>>(p);
            else if (mode == 3 && apply) bn_relu_bwd_kernel<T, 3, true, true><<<grid, kBnThreads, 0, stream>>>(p);
            else if (mode == 3) bn_relu_bwd_kernel<T, 3, false, true><<<grid, kBnThreads, 0, stream>>>(p);
            else if (apply) bn_relu_bwd_kernel<T, 0, true, true><<<grid, kBnThreads, 0, stream>>>(p);
            else bn_relu_bwd_kernel<T, 0, false, true><<<grid, kBnThreads, 0, stream>>>(p);
        }
        else if (mode == 1 && apply) bn_relu_bwd_kernel<T, 1, true, false><<<grid, kBnThreads, 0, stream>>>(p);
        else if (mode == 1) bn_relu_bwd_kernel<T, 1, false, false><<<grid, kBnThreads, 0, stream>>>(p);
        else if (mode == 2 && apply) bn_relu_bwd_kernel<T, 2, true, false><<<grid, kBnThreads, 0, stream>>>(p);
        else if (mode == 2) bn_relu_bwd_kernel<T, 2, false, false><<<grid, kBnThreads, 0, stream>>>(p);
        else if (mode == 3 && apply) bn_relu_bwd_kernel<T, 3, true, false><<<grid, kBnThreads, 0, stream>>>(p);
        else if (mode == 3) bn_relu_bwd_kernel<T, 3, false, false><<<grid, kBnThreads, 0, stream>>>(p);
        else if (apply) bn_relu_bwd_kernel<T, 0, true, false><<<grid, kBnThreads, 0, stream>>>(p);
        else bn_relu_bwd_kernel<T, 0, false, false><<<grid, kBnThreads, 0, stream>>>(p);
    });
    return check_launch(what);
}

int ctu_bn_relu_bwd_reduce_drop(int dtype, const void* y, const float* ss, const void* dA, const void* dP, double* sums2,
                                int c, int n, int d, int h, int w, int y_phase_major, const float* keep, ctu_stream stream) {
    const char* what = keep ? "ctu_bn_relu_bwd_reduce_drop" : "ctu_bn_relu_bwd_reduce";
    const bool prezeroed = (y_phase_major & CTU_ACCUM_PREZEROED) != 0;
    y_phase_major &= ~CTU_ACCUM_PREZEROED;
    CTU_REQUIRE(y && ss && sums2 && (dA || dP) && c > 0 && n > 0 && d > 0 && h > 0 && w > 0, "%s: bad arguments", what);
    BwdArgs p = {};
    p.y = y; p.ss = ss; p.dA = dA; p.dP = dP; p.sums2 = sums2; p.c = c; p.cb = (c + 7) / 8; p.d = d; p.h = h; p.w = w;
    p.keep = keep;
    cudaError_t e = prezeroed ? cudaSuccess : cudaMemsetAsync(sums2, 0, sizeof(double) * 2 * p.cb * 8, (cudaStream_t)stream);
    if (e != cudaSuccess) {
        set_error("%s: memset: %s", what, cudaGetErrorString(e));
        return (int)e;
    }
    return bn_bwd(dtype, p, n, false, y_phase_major, (cudaStream_t)stream, what);
}

int ctu_bn_relu_bwd_reduce(int dtype, const void* y, const float* ss, const void* dA, const void* dP, double* sums2,
                           int c, int n, int d, int h, int w, int y_phase_major, ctu_stream stream) {
    return ctu_bn_relu_bwd_reduce_drop(dtype, y, ss, dA, dP, sums2, c, n, d, h, w, y_phase_major, nullptr, stream);
}

int ctu_bn_relu_bwd_apply_drop(int dtype, const void* y, const float* ss, const float* gamma, const void* dA, const void* dP,
                               const double* sums2, double count, void* dy, float* dgamma, float* dbeta, int c, int n, int d,
                               int h, int w, int y_phase_major, const float* keep, ctu_stream stream) {
    const char* what = keep ? "ctu_bn_relu_bwd_apply_drop" : "ctu_bn_relu_bwd_apply";
    CTU_REQUIRE(y && ss && sums2 && dy && dgamma && dbeta && (dA || dP) && count > 0 && c > 0 && n > 0 && d > 0 && h > 0 && w > 0,
                "%s: bad arguments", what);
    BwdArgs p = {};
    p.y = y; p.ss = ss; p.gamma = gamma; p.dA = dA; p.dP = dP; p.sums2 = const_cast<double*>(sums2); p.count = count;
    p.dy = dy; p.dgamma = dgamma; p.dbeta = dbeta; p.c = c; p.cb = (c + 7) / 8; p.d = d; p.h = h; p.w = w;
    p.keep = keep;
    return bn_bwd(dtype, p, n, true, y_phase_major, (cudaStream_t)stream, what);
}

int ctu_bn_relu_bwd_apply(int dtype, const void* y, const float* ss, const float* gamma, const void* dA, const void* dP,
                          const double* sums2, double count, void* dy, float* dgamma, float* dbeta, int c, int n, int d,
                          int h, int w, int y_phase_major, ctu_stream stream) {
    return ctu_bn_relu_bwd_apply_drop(dtype, y, ss, gamma, dA, dP, sums2, count, dy, dgamma, dbeta, c, n, d, h, w,
                                      y_phase_major, nullptr, stream);
}

}  // extern "C"
