// Error plumbing, activation layout conversion and weight (un)packing.
#include "common.cuh"

namespace ctu {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: %s", what, cudaGetErrorString(e));
        return (int)e;
    }
    return CTU_OK;
}

// ---------------------------------------------------------------- activations
// fp32 NCDHW -> blocked [N][Cb][S][8].  One thread per (n, cb, voxel): reads 8 planes (each read
// coalesced across the warp), writes one 16/32-byte group.
template <typename T>
__global__ void pack_kernel(const float* __restrict__ src, T* __restrict__ dst, int c, int cb, long long spatial,
                            long long total) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    long long s = i % spatial;
    long long ncb = i / spatial;
    int b = (int)(ncb % cb);
    long long n = ncb / cb;
    V8 r;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        int ch = b * 8 + j;
        r.v[j] = ch < c ? __ldg(src + (n * c + ch) * spatial + s) : 0.f;
    }
    Vec8<T>::store(dst + i * 8, r);
}

// four consecutive voxels per thread (spatial % 4 == 0): one 16-byte load per real channel, four group stores
template <typename T>
__global__ void pack4_kernel(const float* __restrict__ src, T* __restrict__ dst, int c, int cb, long long spatial4,
                             long long total4) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total4) return;
    const long long s4 = i % spatial4;
    const long long ncb = i / spatial4;
    const int b = (int)(ncb % cb);
    const long long n = ncb / cb, spatial = spatial4 * 4;
    float4 v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int ch = b * 8 + j;
        v[j] = ch < c ? __ldg(reinterpret_cast<const float4*>(src + (n * c + ch) * spatial) + s4) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    T* out = dst + (ncb * spatial + s4 * 4) * 8;
    V8 r;
#pragma unroll
    for (int j = 0; j < 8; ++j) r.v[j] = v[j].x;
    Vec8<T>::store(out, r);
#pragma unroll
    for (int j = 0; j < 8; ++j) r.v[j] = v[j].y;
    Vec8<T>::store(out + 8, r);
#pragma unroll
    for (int j = 0; j < 8; ++j) r.v[j] = v[j].z;
    Vec8<T>::store(out + 16, r);
#pragma unroll
    for (int j = 0; j < 8; ++j) r.v[j] = v[j].w;
    Vec8<T>::store(out + 24, r);
}

// Patch gather for sliding-window inference: B patches of p^3 voxels out of a float32 [C][D][H][W] volume at the origins
// listed in device memory -> blocked [B][Cb][p][p][p][8].  Four x-consecutive voxels per thread (16-byte loads per channel).
// A patch that lies inside the volume with a 16-byte aligned x origin (vec4: the volume width is a multiple of 4 and the
// volume is 16-byte aligned) takes the float4 loads; any other window -- an origin anywhere, a width that is not a
// multiple of 4, a window reaching past a face -- reads voxel by voxel and zero-fills whatever lies outside the volume.
// The origins are device data, so the choice is made per patch here.
template <typename T>
__global__ void pack_patches_kernel(const float* __restrict__ vol, const int* __restrict__ origins, T* __restrict__ dst, int c,
                                    int cb, int D, int H, int W, int p, long long total4, int vec4) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total4) return;
    const int p4 = p >> 2;
    const int x4 = (int)(i % p4);
    long long r = i / p4;
    const int y = (int)(r % p); r /= p;
    const int z = (int)(r % p); r /= p;
    const int b = (int)(r % cb);
    const int n = (int)(r / cb);
    const int oz = origins[3 * n], oy = origins[3 * n + 1], ox = origins[3 * n + 2];
    const long long plane = (long long)D * H * W;
    float4 v[8];
    const bool inside = oz >= 0 && oy >= 0 && ox >= 0 && oz + p <= D && oy + p <= H && ox + p <= W;
    if (vec4 && inside && (ox & 3) == 0) {
        const long long src0 = ((long long)(oz + z) * H + (oy + y)) * W + ox + 4 * x4;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int ch = b * 8 + j;
            v[j] = ch < c ? __ldg(reinterpret_cast<const float4*>(vol + ch * plane + src0)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    } else {
        const int gz = oz + z, gy = oy + y, gx = ox + 4 * x4;
        const bool row = gz >= 0 && gz < D && gy >= 0 && gy < H;
        const long long src0 = ((long long)gz * H + gy) * W + gx;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int ch = b * 8 + j;
            float e[4];
#pragma unroll
            for (int k = 0; k < 4; ++k)
                e[k] = (ch < c && row && gx + k >= 0 && gx + k < W) ? __ldg(vol + ch * plane + src0 + k) : 0.f;
            v[j] = make_float4(e[0], e[1], e[2], e[3]);
        }
    }
    T* out = dst + (((((long long)n * cb + b) * p + z) * p + y) * p + 4 * x4) * 8;
    V8 q;
#pragma unroll
    for (int j = 0; j < 8; ++j) q.v[j] = v[j].x;
    Vec8<T>::store(out, q);
#pragma unroll
    for (int j = 0; j < 8; ++j) q.v[j] = v[j].y;
    Vec8<T>::store(out + 8, q);
#pragma unroll
    for (int j = 0; j < 8; ++j) q.v[j] = v[j].z;
    Vec8<T>::store(out + 16, q);
#pragma unroll
    for (int j = 0; j < 8; ++j) q.v[j] = v[j].w;
    Vec8<T>::store(out + 24, q);
}

template <typename T>
__global__ void unpack_kernel(const T* __restrict__ src, float* __restrict__ dst, int c, int cb, long long spatial,
                              long long total) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    long long s = i % spatial;
    long long ncb = i / spatial;
    int b = (int)(ncb % cb);
    long long n = ncb / cb;
    V8 r = Vec8<T>::load(src + i * 8);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        int ch = b * 8 + j;
        if (ch < c) dst[(n * c + ch) * spatial + s] = r.v[j];
    }
}

// ---------------------------------------------------------------- conv weights
// Packed forward layout: wp[((cob*cb_total + cib)*taps + tap)*64 + ci*8 + co].
// `transposed_native` selects ConvTranspose3d's native [Cin][Cout][taps] parameter layout.
// mode 0: pack   (native -> packed), pad entries written as 0
// mode 1: unpack (packed -> native), gradient direction
__global__ void conv_weight_kernel(float* __restrict__ native, float* __restrict__ packed, SrcMap m, int cout, int taps,
                                   int transposed_native, int mode, long long total) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    int co = (int)(i & 7), ci = (int)((i >> 3) & 7);
    long long r = i >> 6;
    int tap = (int)(r % taps);
    r /= taps;
    int cib = (int)(r % m.cb_total);
    int cob = (int)(r / m.cb_total);
    int s = 0;
#pragma unroll
    for (int q = 1; q < CTU_MAX_SRC; ++q)
        if (q < m.nsrc && cib >= m.cboff[q]) s = q;
    int cl = (cib - m.cboff[s]) * 8 + ci;
    int cog = cob * 8 + co;
    bool valid = cl < m.ch[s] && cog < cout;
    long long nidx = 0;
    if (valid) {
        int cig = m.choff[s] + cl;
        nidx = transposed_native ? ((long long)cig * cout + cog) * taps + tap : ((long long)cog * m.c_total + cig) * taps + tap;
    }
    if (mode == 0)
        packed[i] = valid ? native[nidx] : 0.f;
    else if (valid)
        native[nidx] = packed[i];
}

// Data-gradient packing for source `which`: a convolution from dy (cout channels, cob_n blocks) to
// d(src) (cs channels, cbs blocks): wpd[((cbs_i*cob_n + cob)*taps + tapf)*64 + co*8 + ci], with
// flipped taps (tapf = taps-1-tap) for Conv3d; ConvTranspose keeps the tap (it is a gather of the
// 2x2x2 children, see convt.cu).
__global__ void conv_weight_dgrad_kernel(const float* __restrict__ native, float* __restrict__ packed, int c_total,
                                         int choff, int cs, int cout, int taps, int transposed_native, int flip,
                                         long long total) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    int ci = (int)(i & 7), co = (int)((i >> 3) & 7);
    long long r = i >> 6;
    int tapf = (int)(r % taps);
    r /= taps;
    int cob_n = (cout + 7) / 8;
    int cob = (int)(r % cob_n);
    int cbs_i = (int)(r / cob_n);
    int cl = cbs_i * 8 + ci;
    int cog = cob * 8 + co;
    int tap = flip ? taps - 1 - tapf : tapf;
    float v = 0.f;
    if (cl < cs && cog < cout) {
        int cig = choff + cl;
        long long nidx = transposed_native ? ((long long)cig * cout + cog) * taps + tap : ((long long)cog * c_total + cig) * taps + tap;
        v = native[nidx];
    }
    packed[i] = v;
}


// ---------------------------------------------------------------------------- batched index gather
// Every weight re-packing of a pass (native fp32 -> packed fp32, -> bf16 UMMA image, data-gradient variants, the
// weight-streaming image) is a fixed permutation + cast of a parameter tensor.  The permutations are computed once per
// layer signature (engine.py runs the packing kernels above on index-valued inputs) and every later pass replays ALL of
// them as jobs of one launch: dst[i] = idx[i] >= 0 ? src[idx[i]] : 0.
constexpr int GATHER_MAX_JOBS = 96;       // 96 x 40 B of kernel parameters
struct GatherJob {
    const float* src;
    void* dst;
    const int* idx;
    long long count;
    int bf16;
};
struct GatherJobs {
    GatherJob j[GATHER_MAX_JOBS];
};

__global__ void __launch_bounds__(256) gather_batch_kernel(const __grid_constant__ GatherJobs jobs) {
    const GatherJob& job = jobs.j[blockIdx.y];
    const long long n8 = job.count >> 3;
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < n8; q += (long long)gridDim.x * blockDim.x) {
        const int4 i0 = __ldg(reinterpret_cast<const int4*>(job.idx) + 2 * q);
        const int4 i1 = __ldg(reinterpret_cast<const int4*>(job.idx) + 2 * q + 1);
        const int id[8] = {i0.x, i0.y, i0.z, i0.w, i1.x, i1.y, i1.z, i1.w};
        V8 v;
#pragma unroll
        for (int e = 0; e < 8; ++e) v.v[e] = id[e] >= 0 ? __ldg(job.src + id[e]) : 0.f;
        if (job.bf16) Vec8<__nv_bfloat16>::store(reinterpret_cast<__nv_bfloat16*>(job.dst) + 8 * q, v);
        else Vec8<float>::store(reinterpret_cast<float*>(job.dst) + 8 * q, v);
    }
}

}  // namespace ctu

using namespace ctu;

extern "C" {

const char* ctu_last_error(void) { return g_err; }
int ctu_version(void) { return 100; }

int ctu_pack_ncdhw(const float* src, void* dst, int dtype, int n, int c, long long spatial, ctu_stream stream) {
    CTU_REQUIRE(src && dst && n > 0 && c > 0 && spatial > 0, "ctu_pack_ncdhw: bad arguments");
    int cb = (c + 7) / 8;
    long long total = (long long)n * cb * spatial;
    if (spatial % 4 == 0 && (reinterpret_cast<uintptr_t>(src) & 15u) == 0) {
        CTU_DISPATCH_DTYPE(dtype, (pack4_kernel<T><<<cdiv(total / 4, 256), 256, 0, (cudaStream_t)stream>>>(src, (T*)dst, c, cb, spatial / 4, total / 4)));
    } else {
        CTU_DISPATCH_DTYPE(dtype, (pack_kernel<T><<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(src, (T*)dst, c, cb, spatial, total)));
    }
    return check_launch("ctu_pack_ncdhw");
}

int ctu_pack_patches(const float* vol, const int* origins, void* dst, int dtype, int n, int c, int vd, int vh, int vw, int patch,
                     ctu_stream stream) {
    CTU_REQUIRE(vol && origins && dst && n > 0 && c > 0 && vd > 0 && vh > 0 && vw > 0, "ctu_pack_patches: bad arguments");
    CTU_REQUIRE(patch > 0 && patch % 4 == 0, "ctu_pack_patches: the patch size must be a multiple of 4");
    const int cb = (c + 7) / 8;
    const long long total4 = (long long)n * cb * patch * patch * (patch / 4);
    const int vec4 = vw % 4 == 0 && (reinterpret_cast<uintptr_t>(vol) & 15u) == 0;
    CTU_DISPATCH_DTYPE(dtype, (pack_patches_kernel<T><<<cdiv(total4, 256), 256, 0, (cudaStream_t)stream>>>(
                                  vol, origins, (T*)dst, c, cb, vd, vh, vw, patch, total4, vec4)));
    return check_launch("ctu_pack_patches");
}

int ctu_unpack_ncdhw(const void* src, float* dst, int dtype, int n, int c, long long spatial, ctu_stream stream) {
    CTU_REQUIRE(src && dst && n > 0 && c > 0 && spatial > 0, "ctu_unpack_ncdhw: bad arguments");
    int cb = (c + 7) / 8;
    long long total = (long long)n * cb * spatial;
    CTU_DISPATCH_DTYPE(dtype, (unpack_kernel<T><<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>((const T*)src, dst, c, cb, spatial, total)));
    return check_launch("ctu_unpack_ncdhw");
}

static long long wpack_floats(int cout, int taps, int nsrc, const int* h_src_channels) {
    SrcMap m;
    if (make_srcmap(m, nsrc, h_src_channels) != CTU_OK || cout < 1) return -1;
    return (long long)((cout + 7) / 8) * m.cb_total * taps * 64;
}

static int pack_generic(float* native, float* packed, int cout, int taps, int nsrc, const int* h_src_channels,
                        int transposed_native, int mode, ctu_stream stream, const char* what) {
    SrcMap m;
    int rc = make_srcmap(m, nsrc, h_src_channels);
    if (rc != CTU_OK) return rc;
    CTU_REQUIRE(native && packed && cout > 0, "%s: bad arguments", what);
    long long total = (long long)((cout + 7) / 8) * m.cb_total * taps * 64;
    conv_weight_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(native, packed, m, cout, taps, transposed_native, mode, total);
    return check_launch(what);
}

static int pack_dgrad_generic(const float* native, float* packed, int cout, int taps, int nsrc,
                              const int* h_src_channels, int which, int transposed_native, int flip,
                              ctu_stream stream, const char* what) {
    SrcMap m;
    int rc = make_srcmap(m, nsrc, h_src_channels);
    if (rc != CTU_OK) return rc;
    CTU_REQUIRE(native && packed && cout > 0 && which >= 0 && which < nsrc, "%s: bad arguments", what);
    int cs = m.ch[which];
    long long total = (long long)((cs + 7) / 8) * ((cout + 7) / 8) * taps * 64;
    conv_weight_dgrad_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(native, packed, m.c_total, m.choff[which], cs, cout, taps, transposed_native, flip, total);
    return check_launch(what);
}

long long ctu_conv_wpack_floats(int cout, int k, int nsrc, const int* h_src_channels) {
    return wpack_floats(cout, k * k * k, nsrc, h_src_channels);
}
int ctu_conv_pack_weight(const float* w, float* wp, int cout, int k, int nsrc, const int* h_src_channels,
                         ctu_stream stream) {
    return pack_generic((float*)w, wp, cout, k * k * k, nsrc, h_src_channels, 0, 0, stream, "ctu_conv_pack_weight");
}
long long ctu_conv_wpack_dgrad_floats(int cout, int k, int src_channels) {
    return (long long)((src_channels + 7) / 8) * ((cout + 7) / 8) * k * k * k * 64;
}
int ctu_conv_pack_weight_dgrad(const float* w, float* wpd, int cout, int k, int nsrc, const int* h_src_channels,
                               int which, ctu_stream stream) {
    return pack_dgrad_generic(w, wpd, cout, k * k * k, nsrc, h_src_channels, which, 0, 1, stream, "ctu_conv_pack_weight_dgrad");
}
int ctu_conv_unpack_wgrad(const float* dwp, float* dw, int cout, int k, int nsrc, const int* h_src_channels,
                          ctu_stream stream) {
    return pack_generic(dw, (float*)dwp, cout, k * k * k, nsrc, h_src_channels, 0, 1, stream, "ctu_conv_unpack_wgrad");
}

long long ctu_convt_wpack_floats(int cout, int nsrc, const int* h_src_channels) {
    return wpack_floats(cout, 8, nsrc, h_src_channels);
}
int ctu_convt_pack_weight(const float* w, float* wp, int cout, int nsrc, const int* h_src_channels, ctu_stream stream) {
    return pack_generic((float*)w, wp, cout, 8, nsrc, h_src_channels, 1, 0, stream, "ctu_convt_pack_weight");
}
long long ctu_convt_wpack_dgrad_floats(int cout, int src_channels) {
    return (long long)((src_channels + 7) / 8) * ((cout + 7) / 8) * 8 * 64;
}
int ctu_convt_pack_weight_dgrad(const float* w, float* wpd, int cout, int nsrc, const int* h_src_channels, int which,
                                ctu_stream stream) {
    return pack_dgrad_generic(w, wpd, cout, 8, nsrc, h_src_channels, which, 1, 0, stream, "ctu_convt_pack_weight_dgrad");
}
int ctu_convt_unpack_wgrad(const float* dwp, float* dw, int cout, int nsrc, const int* h_src_channels,
                           ctu_stream stream) {
    return pack_generic(dw, (float*)dwp, cout, 8, nsrc, h_src_channels, 1, 1, stream, "ctu_convt_unpack_wgrad");
}

int ctu_gather_batch(int njobs, const float* const* h_srcs, void* const* h_dsts, const int* const* h_idxs,
                     const long long* h_counts, const int* h_dst_bf16, ctu_stream stream) {
    CTU_REQUIRE(njobs > 0 && h_srcs && h_dsts && h_idxs && h_counts && h_dst_bf16, "ctu_gather_batch: bad arguments");
    for (int j0 = 0; j0 < njobs; j0 += GATHER_MAX_JOBS) {
        const int nj = (njobs - j0) < GATHER_MAX_JOBS ? (njobs - j0) : GATHER_MAX_JOBS;
        GatherJobs jobs = {};
        long long most = 0;
        for (int j = 0; j < nj; ++j) {
            GatherJob& g = jobs.j[j];
            g.src = h_srcs[j0 + j]; g.dst = h_dsts[j0 + j]; g.idx = h_idxs[j0 + j]; g.count = h_counts[j0 + j];
            g.bf16 = h_dst_bf16[j0 + j];
            CTU_REQUIRE(g.src && g.dst && g.idx && g.count > 0 && g.count % 8 == 0, "ctu_gather_batch: bad job %d", j0 + j);
            most = g.count > most ? g.count : most;
        }
        long long gx = cdiv(most / 8, 256);
        if (gx > 148 * 8) gx = 148 * 8;
        gather_batch_kernel<<<dim3((unsigned)gx, nj), 256, 0, (cudaStream_t)stream>>>(jobs);
        int rc = check_launch("ctu_gather_batch");
        if (rc != CTU_OK) return rc;
    }
    return CTU_OK;
}

}  // extern "C"
