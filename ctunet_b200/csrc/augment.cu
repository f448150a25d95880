// Salt-and-pepper noise on binary uint8 volumes (the second stage of `flap_rec_transform`).
//   SaltAndPepper.__call__   ctunet/pytorch/transforms.py:13-49
// Per volume: black = (u_b > density * (1 - salt_ratio)), white = 1 - (u_w > density * salt_ratio),
// out = (img AND black) OR white, with u_b, u_w two independent uniform [0, 1) float64 fields.
// The reference draws the fields from numpy's global MT19937 stream on the host (two float64 per voxel); here they come
// from a counter-based Philox4x32-10 generator (one call per voxel = 128 bits = two 53-bit doubles built the way numpy builds
// them: (a >> 5) * 2^26 + (b >> 6)) / 2^53), or from caller-supplied fields -- which makes the mask logic bit-comparable with
// the reference.  The scalar draws (the self-decaying `noise_density`, transforms.py:31, and the per-image gate, :33-34) stay
// on the host RNGs in the reference's order (utilities.SaltAndPepper).
#include "common.cuh"

namespace ctu {

// (philox4x32_10: common.cuh)
__device__ __forceinline__ double u53(uint32_t a, uint32_t b) {
    return ((double)(a >> 5) * 67108864.0 + (double)(b >> 6)) / 9007199254740992.0;
}

__global__ void __launch_bounds__(256) salt_pepper_kernel(const unsigned char* __restrict__ img, unsigned char* __restrict__ out,
                                                          long long nvox, double thr_black, double thr_white,
                                                          const double* __restrict__ ub, const double* __restrict__ uw,
                                                          unsigned long long seed, unsigned long long offset) {
    for (long long v = (long long)blockIdx.x * 256 + threadIdx.x; v < nvox; v += (long long)gridDim.x * 256) {
        double b, w;
        if (ub) {
            b = ub[v];
            w = uw[v];
        } else {
            const unsigned long long ctr = offset + (unsigned long long)v;
            uint32_t c[4] = {(uint32_t)ctr, (uint32_t)(ctr >> 32), 0u, 0u};
            philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
            b = u53(c[0], c[1]);
            w = u53(c[2], c[3]);
        }
        const bool black = b > thr_black;          // 1 keeps the voxel, 0 = pepper
        const bool white = !(w > thr_white);       // 1 = salt
        out[v] = (unsigned char)(((img[v] != 0) && black) || white);
    }
}

}  // namespace ctu

using namespace ctu;

extern "C" int ctu_salt_pepper_u8(const unsigned char* img, unsigned char* out, long long nvox, double noise_density,
                                  double salt_ratio, const double* u_black, const double* u_white, unsigned long long seed,
                                  unsigned long long offset, ctu_stream stream) {
    CTU_REQUIRE(img && out && nvox >= 1, "ctu_salt_pepper_u8: null pointer / empty volume");
    CTU_REQUIRE((u_black == nullptr) == (u_white == nullptr), "ctu_salt_pepper_u8: supply both uniform fields or neither");
    const int blocks = (int)min((long long)148 * 16, (nvox + 255) / 256);
    salt_pepper_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(img, out, nvox, noise_density * (1 - salt_ratio),
                                                                 noise_density * salt_ratio, u_black, u_white, seed, offset);
    return check_launch("salt_pepper_kernel");
}

// Random affine augmentation of mask batches (no reference counterpart: the reference has no spatial augmentation;
// DESIGN.md section 7e).  Per sample one map from output voxel p = (z, y, x) to source point
//   q = c + t + (1/s) R F (p - c),  c = (S - 1) / 2,  R = R_d(a_d) R_h(a_h) R_w(a_w),  F = diag(+-1)
// stored as a float32 matrix M [3][4] (built in double, rounded once).  Nearest neighbour, in float32 in exactly this order
// with no contraction:  q_k = ((M_k0 z + M_k1 y) + M_k2 x) + M_k3,  i_k = floor(q_k + 0.5);  a source outside the volume
// (tested in float, so NaN / inf coordinates fail it) reads 0.  Every mask of a sample uses the same index, which keeps
// broken & flap == 0 and broken | flap == full exact.
namespace ctu {

constexpr int kAffineThreads = 256;
constexpr int kAffineRun = 16;             // consecutive x voxels per thread

struct AffineRanges {
    float rot[3];                          // max |angle| about d, h, w, radians
    float scale_lo, scale_hi;
    float trans[3];                        // max |translation| along z, y, x, voxels
    int flip;                              // bit k: axis k may flip
};

__device__ __forceinline__ float u24(uint32_t r) { return (float)(r >> 8) * (1.f / 16777216.f); }

// One single-block launch per batch: params [b][10] = (a_d, a_h, a_w, s, t_z, t_y, t_x, f_z, f_y, f_x), matrices [b][12].
// Philox4x32-10 with counter = (pass, sample, call), key = seed; the pass number is read by every thread before the
// barrier behind which thread 0 advances it (the protocol of dropout3d_keep_kernel).
__global__ void __launch_bounds__(kAffineThreads) affine_draw_kernel(AffineRanges rg, int batch, int d, int h, int w,
                                                                     unsigned long long key,
                                                                     unsigned long long* pass_counter,
                                                                     float* __restrict__ params, float* __restrict__ mats) {
    const unsigned long long pass = pass_counter != nullptr ? *pass_counter : 0ull;
    __syncthreads();
    if (threadIdx.x == 0 && pass_counter != nullptr) *pass_counter = pass + 1;
    for (int i = threadIdx.x; i < batch; i += kAffineThreads) {
        float u[12];
#pragma unroll
        for (int call = 0; call < 3; ++call) {
            uint32_t r[4] = {(uint32_t)pass, (uint32_t)(pass >> 32), (uint32_t)i, (uint32_t)call};
            philox4x32_10(r, (uint32_t)key, (uint32_t)(key >> 32));
#pragma unroll
            for (int j = 0; j < 4; ++j) u[4 * call + j] = u24(r[j]);
        }
        float p[10];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            p[k] = __fmul_rn(rg.rot[k], __fsub_rn(__fmul_rn(2.f, u[k]), 1.f));
            p[4 + k] = __fmul_rn(rg.trans[k], __fsub_rn(__fmul_rn(2.f, u[4 + k]), 1.f));
            p[7 + k] = (((rg.flip >> k) & 1) && u[7 + k] < 0.5f) ? -1.f : 1.f;
        }
        p[3] = __fadd_rn(rg.scale_lo, __fmul_rn(__fsub_rn(rg.scale_hi, rg.scale_lo), u[3]));
#pragma unroll
        for (int k = 0; k < 10; ++k) params[10 * i + k] = p[k];

        double cs[3], sn[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) sincos((double)p[k], &sn[k], &cs[k]);
        const double rd[3][3] = {{1, 0, 0}, {0, cs[0], -sn[0]}, {0, sn[0], cs[0]}};
        const double rh[3][3] = {{cs[1], 0, sn[1]}, {0, 1, 0}, {-sn[1], 0, cs[1]}};
        const double rw[3][3] = {{cs[2], -sn[2], 0}, {sn[2], cs[2], 0}, {0, 0, 1}};
        double t[3][3], a[3][3];
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int c = 0; c < 3; ++c) t[r][c] = rd[r][0] * rh[0][c] + rd[r][1] * rh[1][c] + rd[r][2] * rh[2][c];
        const double inv_s = 1.0 / (double)p[3];
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int c = 0; c < 3; ++c)
                a[r][c] = (t[r][0] * rw[0][c] + t[r][1] * rw[1][c] + t[r][2] * rw[2][c]) * (double)p[7 + c] * inv_s;
        const double ctr[3] = {0.5 * (d - 1), 0.5 * (h - 1), 0.5 * (w - 1)};
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const double off = ctr[r] + (double)p[4 + r] - (a[r][0] * ctr[0] + a[r][1] * ctr[1] + a[r][2] * ctr[2]);
            mats[12 * i + 4 * r] = (float)a[r][0];
            mats[12 * i + 4 * r + 1] = (float)a[r][1];
            mats[12 * i + 4 * r + 2] = (float)a[r][2];
            mats[12 * i + 4 * r + 3] = (float)off;
        }
    }
}

struct AffineIO {
    const unsigned char* src[3];           // uint8 [b][spatial] or bits [b * spatial / 8] (one bit stream for the batch)
    unsigned char* dst[3];                 // uint8 [b][spatial]; with IMAGE, src[0] goes to the image instead of dst[0]
    const float* atlas;                    // [spatial], copied into image channel 1 when cin == 2
    float* image;                          // [b][cin][spatial]
    const float* mat;                      // [b][12]
    int nsrc, cin, d, h, w, runs_per_row;
    long long spatial;
};

// One thread per run of kAffineRun consecutive x voxels of one row: the row term M_k0 z + M_k1 y once per run.  VEC (w a
// multiple of 16, 16-byte aligned buffers) stores with 16-byte vectors like the plain encoders; otherwise voxel by voxel.
template <bool BITS, bool IMAGE, bool VEC>
__global__ void __launch_bounds__(kAffineThreads) affine_gather_kernel(AffineIO a) {
    const int b = blockIdx.y;
    const long long g = (long long)blockIdx.x * kAffineThreads + threadIdx.x;
    const long long row = g / a.runs_per_row;
    if (row >= (long long)a.d * a.h) return;
    const int x0 = (int)(g - row * a.runs_per_row) * kAffineRun;
    const int y = (int)(row % a.h), z = (int)(row / a.h);
    const float* m = a.mat + 12 * b;
    float rt[3], mx[3], mt[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        rt[k] = __fadd_rn(__fmul_rn(__ldg(m + 4 * k), (float)z), __fmul_rn(__ldg(m + 4 * k + 1), (float)y));
        mx[k] = __ldg(m + 4 * k + 2);
        mt[k] = __ldg(m + 4 * k + 3);
    }
    const float lim[3] = {(float)a.d - 0.5f, (float)a.h - 0.5f, (float)a.w - 0.5f};
    const long long base = (long long)b * a.spatial;
    const int n = VEC ? kAffineRun : min(kAffineRun, a.w - x0);
    const long long v0 = ((long long)z * a.h + y) * a.w + x0;
    float* img = IMAGE ? a.image + (long long)b * a.cin * a.spatial + v0 : nullptr;
    const float* atl = IMAGE ? a.atlas + v0 : nullptr;
    uint32_t val[3][4] = {{0u, 0u, 0u, 0u}, {0u, 0u, 0u, 0u}, {0u, 0u, 0u, 0u}};     // VEC: 16 packed bytes per mask
#pragma unroll
    for (int j = 0; j < kAffineRun; ++j) {
        if (!VEC && j >= n) break;
        const float x = (float)(x0 + j);
        float q[3];
        bool in = true;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            q[k] = __fadd_rn(__fadd_rn(rt[k], __fmul_rn(mx[k], x)), mt[k]);
            in = in && q[k] > -0.5f && q[k] < lim[k];
        }
        uint32_t byte[3] = {0u, 0u, 0u};
        if (in) {
            const long long iz = (long long)floorf(__fadd_rn(q[0], 0.5f));
            const int iy = (int)floorf(__fadd_rn(q[1], 0.5f)), ix = (int)floorf(__fadd_rn(q[2], 0.5f));
            const long long v = base + (iz * a.h + iy) * a.w + ix;
#pragma unroll
            for (int s = 0; s < 3; ++s) {
                if (s >= a.nsrc) break;
                byte[s] = BITS ? (uint32_t)(__ldg(a.src[s] + (v >> 3)) >> (v & 7)) & 1u : (uint32_t)__ldg(a.src[s] + v);
            }
        }
        if (VEC) {
#pragma unroll
            for (int s = 0; s < 3; ++s) val[s][j >> 2] |= byte[s] << (8 * (j & 3));
        } else {
            if (IMAGE) {
                img[j] = (float)byte[0];
                if (a.cin > 1) img[a.spatial + j] = atl[j];
            }
#pragma unroll
            for (int s = IMAGE ? 1 : 0; s < 3; ++s)
                if (s < a.nsrc) a.dst[s][base + v0 + j] = (unsigned char)byte[s];
        }
    }
    if (!VEC) return;
    if (IMAGE) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const uint32_t wd = val[0][i];
            *reinterpret_cast<float4*>(img + 4 * i) = make_float4((float)(wd & 0xffu), (float)((wd >> 8) & 0xffu),
                                                                  (float)((wd >> 16) & 0xffu), (float)(wd >> 24));
            if (a.cin > 1) *reinterpret_cast<float4*>(img + a.spatial + 4 * i) = *reinterpret_cast<const float4*>(atl + 4 * i);
        }
    }
#pragma unroll
    for (int s = IMAGE ? 1 : 0; s < 3; ++s)
        if (s < a.nsrc) *reinterpret_cast<uint4*>(a.dst[s] + base + v0) = make_uint4(val[s][0], val[s][1], val[s][2], val[s][3]);
}

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// axes below 2^22: floor(q + 0.5f) of an in-bounds q then stays below the axis length (the float spacing is < 0.5 there)
static inline bool affine_shape_ok(int batch, int d, int h, int w) {
    return batch >= 1 && batch <= 65535 && d >= 1 && h >= 1 && w >= 1 && d < (1 << 22) && h < (1 << 22) && w < (1 << 22);
}

template <bool BITS, bool IMAGE>
static int launch_affine_gather(const AffineIO& io, int batch, cudaStream_t st) {
    bool vec = io.w % kAffineRun == 0;
    for (int s = 0; s < io.nsrc; ++s) vec = vec && (IMAGE && s == 0 ? true : aligned16(io.dst[s]));
    if (IMAGE) vec = vec && aligned16(io.image) && (io.cin == 1 || aligned16(io.atlas));
    const dim3 grid(cdiv((long long)io.d * io.h * io.runs_per_row, kAffineThreads), batch);
    if (vec) affine_gather_kernel<BITS, IMAGE, true><<<grid, kAffineThreads, 0, st>>>(io);
    else affine_gather_kernel<BITS, IMAGE, false><<<grid, kAffineThreads, 0, st>>>(io);
    return CTU_OK;
}

}  // namespace ctu

extern "C" int ctu_affine_draw(int batch, int d, int h, int w, const float* h_ranges, int flip_axes, unsigned long long seed,
                               unsigned long long* pass_counter, float* params, float* matrices, ctu_stream stream) {
    CTU_REQUIRE(affine_shape_ok(batch, d, h, w) && h_ranges && params && matrices && flip_axes >= 0 && flip_axes <= 7,
                "ctu_affine_draw: bad arguments (batch %d, shape %d x %d x %d, flip_axes %d)", batch, d, h, w, flip_axes);
    AffineRanges rg;
    for (int k = 0; k < 3; ++k) {
        rg.rot[k] = h_ranges[k];
        rg.trans[k] = h_ranges[5 + k];
        CTU_REQUIRE(rg.rot[k] >= 0.f && rg.rot[k] <= 3.14159265f && rg.trans[k] >= 0.f && rg.trans[k] <= 1e6f,
                    "ctu_affine_draw: rotation (%g) must be in [0, pi], translation (%g) in [0, 1e6]", (double)rg.rot[k],
                    (double)rg.trans[k]);
    }
    rg.scale_lo = h_ranges[3];
    rg.scale_hi = h_ranges[4];
    CTU_REQUIRE(rg.scale_lo > 0.f && rg.scale_lo <= rg.scale_hi && rg.scale_hi <= 1e3f,
                "ctu_affine_draw: scale range [%g, %g]", (double)rg.scale_lo, (double)rg.scale_hi);
    rg.flip = flip_axes;
    affine_draw_kernel<<<1, kAffineThreads, 0, (cudaStream_t)stream>>>(rg, batch, d, h, w, seed, pass_counter, params, matrices);
    return check_launch("ctu_affine_draw");
}

extern "C" int ctu_affine_encode_flaprec(int bits, const unsigned char* broken, const unsigned char* full,
                                         const unsigned char* flap, const float* atlas, const float* matrices, float* image,
                                         unsigned char* full_mask, unsigned char* flap_mask, int batch, int in_channels, int d,
                                         int h, int w, ctu_stream stream) {
    CTU_REQUIRE(affine_shape_ok(batch, d, h, w) && (bits == 0 || bits == 1),
                "ctu_affine_encode_flaprec: bad arguments (bits %d, batch %d, shape %d x %d x %d)", bits, batch, d, h, w);
    CTU_REQUIRE(broken && full && flap && matrices && image && full_mask && flap_mask,
                "ctu_affine_encode_flaprec: null pointer");
    CTU_REQUIRE(in_channels == 1 || (in_channels == 2 && atlas),
                "ctu_affine_encode_flaprec: 1 input channel, or 2 with an atlas");
    AffineIO io = {};
    io.src[0] = broken, io.src[1] = full, io.src[2] = flap;
    io.dst[1] = full_mask, io.dst[2] = flap_mask;
    io.atlas = atlas, io.image = image, io.mat = matrices;
    io.nsrc = 3, io.cin = in_channels, io.d = d, io.h = h, io.w = w, io.runs_per_row = cdiv(w, kAffineRun);
    io.spatial = (long long)d * h * w;
    cudaStream_t st = (cudaStream_t)stream;
    if (bits) launch_affine_gather<true, true>(io, batch, st);
    else launch_affine_gather<false, true>(io, batch, st);
    return check_launch("ctu_affine_encode_flaprec");
}

extern "C" int ctu_affine_masks_u8(int n, const unsigned char* const* h_src, unsigned char* const* h_dst,
                                   const float* matrices, int batch, int d, int h, int w, ctu_stream stream) {
    CTU_REQUIRE(n >= 1 && n <= 3 && h_src && h_dst && matrices && affine_shape_ok(batch, d, h, w),
                "ctu_affine_masks_u8: bad arguments (n %d, batch %d, shape %d x %d x %d)", n, batch, d, h, w);
    AffineIO io = {};
    for (int s = 0; s < n; ++s) {
        CTU_REQUIRE(h_src[s] && h_dst[s], "ctu_affine_masks_u8: mask %d: null pointer", s);
        io.src[s] = h_src[s];
        io.dst[s] = h_dst[s];
    }
    io.mat = matrices;
    io.nsrc = n, io.cin = 0, io.d = d, io.h = h, io.w = w, io.runs_per_row = cdiv(w, kAffineRun);
    io.spatial = (long long)d * h * w;
    launch_affine_gather<false, false>(io, batch, (cudaStream_t)stream);
    return check_launch("ctu_affine_masks_u8");
}
