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
    const float* mat;                      // [b][12]; NULL in hole mode: the direct index
    const double* hole;                    // hole mode: craniectomy params [b][7] (ctu_craniectomy_draw)
    int nsrc, cin, d, h, w, runs_per_row;
    long long spatial;
};

// One thread per run of kAffineRun consecutive x voxels of one row: the row term M_k0 z + M_k1 y once per run.  VEC (w a
// multiple of 16, 16-byte aligned buffers) stores with 16-byte vectors like the plain encoders; otherwise voxel by voxel.
// HOLE (the virtual craniectomy, DESIGN.md section 7f): src[0] is the full skull only; the source voxel s of output voxel p
// gives full = (src[0][s] != 0), inside = applied && inside(s), and the three values (full AND NOT inside, full,
// full AND inside) take the places of the three gathered masks.  AFFINE = false (no matrices): s = p, the run's 16
// source voxels in one load when VEC.
template <bool BITS, bool IMAGE, bool VEC, bool HOLE = false, bool AFFINE = true>
__global__ void __launch_bounds__(kAffineThreads) affine_gather_kernel(AffineIO a) {
    const int b = blockIdx.y;
    const long long g = (long long)blockIdx.x * kAffineThreads + threadIdx.x;
    const long long row = g / a.runs_per_row;
    if (row >= (long long)a.d * a.h) return;
    const int x0 = (int)(g - row * a.runs_per_row) * kAffineRun;
    const int y = (int)(row % a.h), z = (int)(row / a.h);
    float rt[3], mx[3], mt[3];
    if (AFFINE) {
        const float* m = a.mat + 12 * b;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            rt[k] = __fadd_rn(__fmul_rn(__ldg(m + 4 * k), (float)z), __fmul_rn(__ldg(m + 4 * k + 1), (float)y));
            mx[k] = __ldg(m + 4 * k + 2);
            mt[k] = __ldg(m + 4 * k + 3);
        }
    }
    const float lim[3] = {(float)a.d - 0.5f, (float)a.h - 0.5f, (float)a.w - 0.5f};
    const long long base = (long long)b * a.spatial;
    const int n = VEC ? kAffineRun : min(kAffineRun, a.w - x0);
    const long long v0 = ((long long)z * a.h + y) * a.w + x0;
    bool applied = false;
    int shape = 0, r = 0, cz = 0, cy = 0, cx = 0;
    FlapHole flap = {};
    uint4 run = make_uint4(0u, 0u, 0u, 0u);
    if (HOLE) {
        const double* hp = a.hole + 7 * b;
        applied = __ldg(hp) != 0.0;
        shape = (int)__ldg(hp + 1);
        const double size = __ldg(hp + 2);
        // int32 is exact here: with axes <= 16384 a squared offset sum is at most 3 * 16383^2 < 28377^2, so clamping the
        // radius at 28378 keeps r * r below 2^31 and changes no test (a larger ball holds every voxel anyway)
        r = (int)fmax(-1.0, fmin(size, 28378.0));
        cz = (int)__ldg(hp + 4), cy = (int)__ldg(hp + 5), cx = (int)__ldg(hp + 6);
        if (shape == 2) flap = flap_hole(a.d, a.h, a.w, cz, cy, cx, size, __ldg(hp + 3));
        if (!AFFINE && applied) {          // direct index: skip the voxel tests of a row the hole does not reach
            if (shape == 2) {
                const double dy = y - flap.ey;
                applied = fabs(z - flap.z0) <= flap.half && (dy * dy <= flap.r2 || fabs(y - flap.qy) <= flap.half);
            } else {
                applied = ball_inside<int>(shape, z - cz, y - cy, 0, r);
            }
        }
        if (!AFFINE && VEC) {
            if (BITS) run.x = __ldg(reinterpret_cast<const unsigned short*>(a.src[0] + ((base + v0) >> 3)));
            else run = __ldg(reinterpret_cast<const uint4*>(a.src[0] + base + v0));
        }
    }
    float* img = IMAGE ? a.image + (long long)b * a.cin * a.spatial + v0 : nullptr;
    const float* atl = IMAGE ? a.atlas + v0 : nullptr;
    uint32_t val[3][4] = {{0u, 0u, 0u, 0u}, {0u, 0u, 0u, 0u}, {0u, 0u, 0u, 0u}};     // VEC: 16 packed bytes per mask
#pragma unroll
    for (int j = 0; j < kAffineRun; ++j) {
        if (!VEC && j >= n) break;
        const float x = (float)(x0 + j);
        float q[3];
        bool in = true;
        if (AFFINE) {
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                q[k] = __fadd_rn(__fadd_rn(rt[k], __fmul_rn(mx[k], x)), mt[k]);
                in = in && q[k] > -0.5f && q[k] < lim[k];
            }
        }
        uint32_t byte[3] = {0u, 0u, 0u};
        if (in) {
            long long iz = z;
            int iy = y, ix = x0 + j;
            if (AFFINE) {
                iz = (long long)floorf(__fadd_rn(q[0], 0.5f));
                iy = (int)floorf(__fadd_rn(q[1], 0.5f)), ix = (int)floorf(__fadd_rn(q[2], 0.5f));
            }
            const long long v = base + (iz * a.h + iy) * a.w + ix;
            if (HOLE) {
                uint32_t f;
                if (!AFFINE && VEC) {
                    const uint32_t* rw = &run.x;
                    f = BITS ? (run.x >> j) & 1u : (uint32_t)(((rw[j >> 2] >> (8 * (j & 3))) & 0xffu) != 0u);
                } else {
                    f = BITS ? (uint32_t)(__ldg(a.src[0] + (v >> 3)) >> (v & 7)) & 1u : (uint32_t)(__ldg(a.src[0] + v) != 0);
                }
                const bool inside = applied && (shape == 2 ? flap_inside(flap, (double)iz, (double)iy, (double)ix)
                                                           : ball_inside<int>(shape, (int)iz - cz, iy - cy, ix - cx, r));
                byte[0] = inside ? 0u : f;
                byte[1] = f;
                byte[2] = inside ? f : 0u;
            } else {
#pragma unroll
                for (int s = 0; s < 3; ++s) {
                    if (s >= a.nsrc) break;
                    byte[s] = BITS ? (uint32_t)(__ldg(a.src[s] + (v >> 3)) >> (v & 7)) & 1u : (uint32_t)__ldg(a.src[s] + v);
                }
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

template <bool BITS, bool IMAGE, bool HOLE = false, bool AFFINE = true>
static int launch_affine_gather(const AffineIO& io, int batch, cudaStream_t st) {
    bool vec = io.w % kAffineRun == 0;
    for (int s = 0; s < io.nsrc; ++s) vec = vec && (IMAGE && s == 0 ? true : aligned16(io.dst[s]));
    if (IMAGE) vec = vec && aligned16(io.image) && (io.cin == 1 || aligned16(io.atlas));
    if (HOLE && !AFFINE) vec = vec && aligned16(io.src[0]);
    const dim3 grid(cdiv((long long)io.d * io.h * io.runs_per_row, kAffineThreads), batch);
    if (vec) affine_gather_kernel<BITS, IMAGE, true, HOLE, AFFINE><<<grid, kAffineThreads, 0, st>>>(io);
    else affine_gather_kernel<BITS, IMAGE, false, HOLE, AFFINE><<<grid, kAffineThreads, 0, st>>>(io);
    return CTU_OK;
}

// ---- virtual craniectomy drawn on the device (DESIGN.md section 7f; the distribution of random_blank_patch(image, p, True,
// p_type="random", valid_shapes), transforms.py:241-300, per sample, with Philox draws instead of the host RNGs).
// Philox4x32-10, key = seed, counter = (pass, sample, call); words r[call][0..3] feed the draws:
//   call 0: u53(r0, r1) gate (applied iff u <= p and the skull is not empty); r2 | r3 << 32 picks the centre
//   call 1: r0 | r1 << 32 the radius, r2 | r3 << 32 the shape
//   call 2: u53(r0, r1) the flap's cylinder radius c_diam = ((0.25 + 0.75 u) * radius) / 4 (utilities.py:146-148)
// A 64-bit word r picks floor(r * n / 2^64) of n choices: the k-th bone voxel in C order (np.argwhere(full > 0)[k]), the
// radius min_r + floor(r * (max_r - min_r) / 2^64), the enabled shape of that rank in the order sphere, box, flap.
constexpr int kHoleChunk = 4096;           // voxels per count chunk: 256 threads x 16
constexpr int kHoleDrawThreads = 1024;

struct HoleDraw {
    double p;
    int shapes;                            // bit 0 sphere, 1 box, 2 flap
    int min_r, n_r;                        // radius in [min_r, min_r + n_r)
};

template <bool BITS>
__device__ __forceinline__ uint32_t bone_at(const unsigned char* __restrict__ m, long long v) {
    return BITS ? (uint32_t)(__ldg(m + (v >> 3)) >> (v & 7)) & 1u : (uint32_t)(__ldg(m + v) != 0);
}

// counts[b][chunk] = bone voxels of the chunk (no atomics, no memset: every CTA writes its own count)
template <bool BITS>
__global__ void __launch_bounds__(256) craniectomy_count_kernel(const unsigned char* __restrict__ full, long long spatial,
                                                                int nchunks, int* __restrict__ counts) {
    const int b = blockIdx.y;
    const long long v0 = (long long)blockIdx.x * kHoleChunk + 16 * threadIdx.x;      // within the sample
    const long long gv = (long long)b * spatial + v0;
    int cnt = 0;
    // fast path: 16 whole voxels behind a naturally aligned 2-byte (bits) or 16-byte (uint8) load; a bit-packed batch
    // whose voxel count is not a multiple of 16, or a view at an odd byte offset, takes the per-byte path
    if (v0 + 16 <= spatial && (BITS ? (gv & 15) == 0 && ((reinterpret_cast<uintptr_t>(full) + (gv >> 3)) & 1) == 0
                                    : ((reinterpret_cast<uintptr_t>(full) + gv) & 15) == 0)) {
        if (BITS) {
            cnt = __popc((uint32_t)__ldg(reinterpret_cast<const unsigned short*>(full + (gv >> 3))));
        } else {
            const uint4 u = __ldg(reinterpret_cast<const uint4*>(full + gv));
            const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
            for (int j = 0; j < 4; ++j)  // a byte is non-zero <=> its low 7 bits carry into bit 7, or bit 7 is set
                cnt += __popc((((w[j] & 0x7f7f7f7fu) + 0x7f7f7f7fu) | w[j]) & 0x80808080u);
        }
    } else {
        for (int j = 0; j < 16 && v0 + j < spatial; ++j) cnt += bone_at<BITS>(full, gv + j);
    }
    __shared__ int red[8];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i) t += red[i];
        counts[(long long)b * nchunks + blockIdx.x] = t;
    }
}

// 32 voxels from global voxel gv as a bit mask (bit i = voxel gv + i is bone), only the first nvalid of them
template <bool BITS>
__device__ __forceinline__ uint32_t bone_word(const unsigned char* __restrict__ m, long long gv, long long nvalid) {
    if (nvalid <= 0) return 0u;
    if (BITS) {
        if (nvalid >= 32 && ((reinterpret_cast<uintptr_t>(m) + (gv >> 3)) & 3) == 0 && (gv & 7) == 0)
            return __ldg(reinterpret_cast<const uint32_t*>(m + (gv >> 3)));
        const long long last = (gv + min(nvalid, 32LL) - 1) >> 3;
        unsigned long long x = 0;
        for (long long i = gv >> 3; i <= last; ++i) x |= (unsigned long long)__ldg(m + i) << (8 * (i - (gv >> 3)));
        x >>= (gv & 7);
        return (uint32_t)x & (nvalid >= 32 ? 0xffffffffu : (1u << nvalid) - 1u);
    }
    if (nvalid >= 32 && ((reinterpret_cast<uintptr_t>(m) + gv) & 15) == 0) {
        uint32_t out = 0;
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const uint4 u = __ldg(reinterpret_cast<const uint4*>(m + gv) + q);
            const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {    // a byte is non-zero <=> its low 7 bits carry into bit 7, or bit 7 is set
                const uint32_t t = ((((w[j] & 0x7f7f7f7fu) + 0x7f7f7f7fu) | w[j]) & 0x80808080u) >> 7;
                out |= ((t | (t >> 7) | (t >> 14) | (t >> 21)) & 0xfu) << (16 * q + 4 * j);
            }
        }
        return out;
    }
    uint32_t out = 0;
    for (int i = 0; i < 32 && i < nvalid; ++i) out |= (uint32_t)(__ldg(m + gv + i) != 0) << i;
    return out;
}

// One CTA for the batch, one warp per sample: params[b][7] = (applied, shape, radius, c_diam, z, y, x); a sample that is
// not applied has centre (-1, -1, -1).  The two-phase search of kth_nonzero_kernel (misc.cu) with k drawn on the device:
// a prefix over the chunk counts (a contiguous range of chunks per lane) finds the chunk, a prefix over its voxels (128
// consecutive voxels per lane, as 32-voxel bit masks) the voxel.  The pass counter is read by every thread before the
// barrier behind which thread 0 advances it (the protocol of affine_draw_kernel).
template <bool BITS>
__global__ void __launch_bounds__(kHoleDrawThreads) craniectomy_draw_kernel(const unsigned char* __restrict__ full, int batch,
                                                                            int d, int h, int w, int nchunks,
                                                                            const int* __restrict__ counts, HoleDraw hd,
                                                                            unsigned long long key,
                                                                            unsigned long long* pass_counter,
                                                                            double* __restrict__ params) {
    const unsigned long long pass = pass_counter != nullptr ? *pass_counter : 0ull;
    __syncthreads();
    if (threadIdx.x == 0 && pass_counter != nullptr) *pass_counter = pass + 1;
    const int lane = threadIdx.x & 31;
    const long long spatial = (long long)d * h * w;
    const int per = (nchunks + 31) / 32;
    const int c0 = min(nchunks, lane * per), c1 = min(nchunks, c0 + per);
    const int n_shapes = __popc(hd.shapes);
    for (int b = threadIdx.x >> 5; b < batch; b += kHoleDrawThreads / 32) {
        uint32_t r[3][4];
#pragma unroll
        for (int call = 0; call < 3; ++call) {
            r[call][0] = (uint32_t)pass, r[call][1] = (uint32_t)(pass >> 32), r[call][2] = (uint32_t)b, r[call][3] = (uint32_t)call;
            philox4x32_10(r[call], (uint32_t)key, (uint32_t)(key >> 32));
        }
        const int* cnt = counts + (long long)b * nchunks;
        long long mine = 0;
        for (int c = c0; c < c1; ++c) mine += __ldg(cnt + c);
        long long inc = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        const long long n = __shfl_sync(0xffffffffu, inc, 31), before = inc - mine;
        const bool applied = u53(r[0][0], r[0][1]) <= hd.p && n > 0;              // uniform over the warp
        double* out = params + 7 * (long long)b;
        if (applied) {
            const long long k = (long long)__umul64hi(r[0][2] | ((unsigned long long)r[0][3] << 32), (unsigned long long)n);
            const bool mine_k = k >= before && k < before + mine;
            long long chunk = 0, rank = 0;
            if (mine_k) {
                long long seen = before;
                for (int c = c0; c < c1; ++c) {
                    const int m = __ldg(cnt + c);
                    if (seen + m > k) {
                        chunk = c;
                        rank = k - seen;
                        break;
                    }
                    seen += m;
                }
            }
            const int owner = __ffs(__ballot_sync(0xffffffffu, mine_k)) - 1;
            chunk = __shfl_sync(0xffffffffu, chunk, owner);
            rank = __shfl_sync(0xffffffffu, rank, owner);
            const long long first = chunk * kHoleChunk + 128LL * lane;            // within the sample
            uint32_t wd[4];
            int cl = 0;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                wd[i] = bone_word<BITS>(full, (long long)b * spatial + first + 32 * i, spatial - first - 32 * i);
                cl += __popc(wd[i]);
            }
            int ci = cl;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, ci, o);
                if (lane >= o) ci += t;
            }
            long long rr = rank - (ci - cl);
            if (rr >= 0 && rr < cl) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int pc = __popc(wd[i]);
                    if (rr < pc) {
                        const long long v = first + 32 * i + __fns(wd[i], 0, (int)rr + 1);
                        out[4] = (double)(v / ((long long)w * h));
                        out[5] = (double)((v / w) % h);
                        out[6] = (double)(v % w);
                        break;
                    }
                    rr -= pc;
                }
            }
        }
        if (lane == 0) {
            const long long radius = hd.min_r + (long long)__umul64hi(r[1][0] | ((unsigned long long)r[1][1] << 32),
                                                                      (unsigned long long)hd.n_r);
            int rank = (int)__umul64hi(r[1][2] | ((unsigned long long)r[1][3] << 32), (unsigned long long)n_shapes);
            int shape = 0;
            for (; shape < 3; ++shape)
                if (((hd.shapes >> shape) & 1) && rank-- == 0) break;
            out[0] = applied ? 1.0 : 0.0;
            out[1] = (double)shape;
            out[2] = (double)radius;
            out[3] = shape == 2 ? __dmul_rn(__dadd_rn(0.25, __dmul_rn(0.75, u53(r[2][0], r[2][1]))), (double)radius) / 4.0 : 0.0;
            if (!applied) out[4] = out[5] = out[6] = -1.0;
        }
    }
}

static inline bool craniectomy_shape_ok(int batch, int d, int h, int w) {
    return batch >= 1 && batch <= 65535 && d >= 1 && h >= 1 && w >= 1 && d <= 16384 && h <= 16384 && w <= 16384;
}

static inline long long craniectomy_ws_bytes(int batch, int d, int h, int w) {
    const long long chunks = cdiv((long long)d * h * w, kHoleChunk);
    return (batch * chunks * (long long)sizeof(int) + 15) / 16 * 16;
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

extern "C" long long ctu_craniectomy_workspace_bytes(int batch, int d, int h, int w) {
    if (!craniectomy_shape_ok(batch, d, h, w)) return -1;
    return craniectomy_ws_bytes(batch, d, h, w);
}

extern "C" int ctu_craniectomy_draw(int bits, const unsigned char* full, int batch, int d, int h, int w, double p,
                                    int shapes, int min_radius, int max_radius, unsigned long long seed,
                                    unsigned long long* pass_counter, double* params, void* ws, long long ws_bytes,
                                    ctu_stream stream) {
    CTU_REQUIRE(craniectomy_shape_ok(batch, d, h, w) && (bits == 0 || bits == 1),
                "ctu_craniectomy_draw: bad arguments (bits %d, batch %d, shape %d x %d x %d)", bits, batch, d, h, w);
    CTU_REQUIRE(full && params && ws && (reinterpret_cast<uintptr_t>(params) & 7u) == 0,
                "ctu_craniectomy_draw: null or misaligned pointer");
    CTU_REQUIRE(p >= 0.0 && p <= 1.0, "ctu_craniectomy_draw: p = %g must be in [0, 1]", p);
    CTU_REQUIRE(shapes >= 1 && shapes <= 7, "ctu_craniectomy_draw: shapes = %d (bit 0 sphere, 1 box, 2 flap)", shapes);
    CTU_REQUIRE(min_radius < max_radius, "ctu_craniectomy_draw: empty radius range [%d, %d)", min_radius, max_radius);
    CTU_REQUIRE(ws_bytes >= craniectomy_ws_bytes(batch, d, h, w) && (reinterpret_cast<uintptr_t>(ws) & 15u) == 0,
                "ctu_craniectomy_draw: workspace of %lld bytes (16-byte aligned, ctu_craniectomy_workspace_bytes)", ws_bytes);
    const long long spatial = (long long)d * h * w;
    const int nchunks = cdiv(spatial, kHoleChunk);
    int* counts = static_cast<int*>(ws);
    const HoleDraw hd = {p, shapes, min_radius, max_radius - min_radius};
    cudaStream_t st = (cudaStream_t)stream;
    const dim3 grid(nchunks, batch);
    if (bits) {
        craniectomy_count_kernel<true><<<grid, 256, 0, st>>>(full, spatial, nchunks, counts);
        craniectomy_draw_kernel<true><<<1, kHoleDrawThreads, 0, st>>>(full, batch, d, h, w, nchunks, counts, hd, seed,
                                                                      pass_counter, params);
    } else {
        craniectomy_count_kernel<false><<<grid, 256, 0, st>>>(full, spatial, nchunks, counts);
        craniectomy_draw_kernel<false><<<1, kHoleDrawThreads, 0, st>>>(full, batch, d, h, w, nchunks, counts, hd, seed,
                                                                       pass_counter, params);
    }
    return check_launch("ctu_craniectomy_draw");
}

extern "C" int ctu_craniectomy_encode_flaprec(int bits, const unsigned char* full, const double* params, const float* atlas,
                                              const float* matrices, float* image, unsigned char* full_mask,
                                              unsigned char* flap_mask, int batch, int in_channels, int d, int h, int w,
                                              ctu_stream stream) {
    CTU_REQUIRE(craniectomy_shape_ok(batch, d, h, w) && (bits == 0 || bits == 1),
                "ctu_craniectomy_encode_flaprec: bad arguments (bits %d, batch %d, shape %d x %d x %d)", bits, batch, d, h, w);
    CTU_REQUIRE(full && params && image && full_mask && flap_mask && (reinterpret_cast<uintptr_t>(params) & 7u) == 0,
                "ctu_craniectomy_encode_flaprec: null or misaligned pointer");
    CTU_REQUIRE(in_channels == 1 || (in_channels == 2 && atlas),
                "ctu_craniectomy_encode_flaprec: 1 input channel, or 2 with an atlas");
    AffineIO io = {};
    io.src[0] = full;
    io.dst[1] = full_mask, io.dst[2] = flap_mask;
    io.atlas = atlas, io.image = image, io.mat = matrices, io.hole = params;
    io.nsrc = 3, io.cin = in_channels, io.d = d, io.h = h, io.w = w, io.runs_per_row = cdiv(w, kAffineRun);
    io.spatial = (long long)d * h * w;
    cudaStream_t st = (cudaStream_t)stream;
    if (matrices) {
        if (bits) launch_affine_gather<true, true, true, true>(io, batch, st);
        else launch_affine_gather<false, true, true, true>(io, batch, st);
    } else {
        if (bits) launch_affine_gather<true, true, true, false>(io, batch, st);
        else launch_affine_gather<false, true, true, false>(io, batch, st);
    }
    return check_launch("ctu_craniectomy_encode_flaprec");
}

extern "C" int ctu_craniectomy_masks_u8(const unsigned char* full, const double* params, unsigned char* broken,
                                        unsigned char* full_out, unsigned char* flap, int batch, int d, int h, int w,
                                        ctu_stream stream) {
    CTU_REQUIRE(craniectomy_shape_ok(batch, d, h, w), "ctu_craniectomy_masks_u8: bad arguments (batch %d, shape %d x %d x %d)",
                batch, d, h, w);
    CTU_REQUIRE(full && params && broken && full_out && flap && (reinterpret_cast<uintptr_t>(params) & 7u) == 0,
                "ctu_craniectomy_masks_u8: null or misaligned pointer");
    AffineIO io = {};
    io.src[0] = full;
    io.dst[0] = broken, io.dst[1] = full_out, io.dst[2] = flap;
    io.hole = params;
    io.nsrc = 3, io.cin = 0, io.d = d, io.h = h, io.w = w, io.runs_per_row = cdiv(w, kAffineRun);
    io.spatial = (long long)d * h * w;
    launch_affine_gather<false, false, true, false>(io, batch, (cudaStream_t)stream);
    return check_launch("ctu_craniectomy_masks_u8");
}
