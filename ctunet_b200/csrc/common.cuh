// Shared device/host helpers for the ctunet_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/ctunet_b200.h"

namespace ctu {

// ---------------------------------------------------------------- error plumbing
void set_error(const char* fmt, ...);
int check_launch(const char* what);

#define CTU_REQUIRE(cond, ...)                 \
    do {                                       \
        if (!(cond)) {                         \
            ctu::set_error(__VA_ARGS__);       \
            return CTU_ERR_INVALID;            \
        }                                      \
    } while (0)

static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

// ---------------------------------------------------------------- 8-channel vectors
// Activations live in a channel-blocked layout [N][Cb][D][H][W][8] (8 channels of one voxel are
// contiguous: 16 B in bf16, 32 B in fp32).  V8 is the register image of one such group.
struct V8 {
    float v[8];
};

template <typename T> struct Vec8;

template <> struct Vec8<float> {
    static __device__ __forceinline__ V8 load(const float* p) {
        V8 r;
        float4 a = *reinterpret_cast<const float4*>(p);
        float4 b = *reinterpret_cast<const float4*>(p + 4);
        r.v[0] = a.x; r.v[1] = a.y; r.v[2] = a.z; r.v[3] = a.w;
        r.v[4] = b.x; r.v[5] = b.y; r.v[6] = b.z; r.v[7] = b.w;
        return r;
    }
    static __device__ __forceinline__ void store(float* p, const V8& r) {
        *reinterpret_cast<float4*>(p) = make_float4(r.v[0], r.v[1], r.v[2], r.v[3]);
        *reinterpret_cast<float4*>(p + 4) = make_float4(r.v[4], r.v[5], r.v[6], r.v[7]);
    }
};

template <> struct Vec8<__nv_bfloat16> {
    static __device__ __forceinline__ V8 load(const __nv_bfloat16* p) {
        V8 r;
        uint4 u = *reinterpret_cast<const uint4*>(p);
        const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            r.v[2 * i] = __uint_as_float(w[i] << 16);
            r.v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
        }
        return r;
    }
    static __device__ __forceinline__ void store(__nv_bfloat16* p, const V8& r) {
        uint32_t w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            __nv_bfloat162 h = __floats2bfloat162_rn(r.v[2 * i], r.v[2 * i + 1]);
            w[i] = *reinterpret_cast<uint32_t*>(&h);
        }
        *reinterpret_cast<uint4*>(p) = make_uint4(w[0], w[1], w[2], w[3]);
    }
};

// Register-frugal staging: keep the 8 channels of a voxel in their STORAGE form (4 registers in bf16) and unpack on use.
template <typename T> struct Raw8;
template <> struct Raw8<float> {
    V8 v;
    __device__ __forceinline__ void load(const float* p) { v = Vec8<float>::load(p); }
    __device__ __forceinline__ V8 get() const { return v; }
};
template <> struct Raw8<__nv_bfloat16> {
    uint4 u;
    __device__ __forceinline__ void load(const __nv_bfloat16* p) { u = *reinterpret_cast<const uint4*>(p); }
    __device__ __forceinline__ V8 get() const {
        V8 r;
        const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            r.v[2 * i] = __uint_as_float(w[i] << 16);
            r.v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
        }
        return r;
    }
};

// 256-bit global accesses (sm_100: LDG/STG.256): two x-adjacent voxels of a bf16 channel block in one instruction.
// The address must be 32-byte aligned.
__device__ __forceinline__ void ldg256(const void* p, uint4& a, uint4& b) {
    asm volatile("ld.global.nc.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w)
                 : "l"(p));
}
__device__ __forceinline__ void stg256(void* p, const uint4& a, const uint4& b) {
    asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w), "r"(b.x),
                 "r"(b.y), "r"(b.z), "r"(b.w)
                 : "memory");
}
__device__ __forceinline__ uint4 pack_bf16x8(const V8& r) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        __nv_bfloat162 h = __floats2bfloat162_rn(r.v[2 * i], r.v[2 * i + 1]);
        w[i] = *reinterpret_cast<uint32_t*>(&h);
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}
__device__ __forceinline__ V8 unpack_bf16x8(const uint4& u) {
    V8 r;
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        r.v[2 * i] = __uint_as_float(w[i] << 16);
        r.v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
    return r;
}

// Value as it will be read back after a store in storage type T (so statistics are taken on what
// the next kernel really sees).
template <typename T> __device__ __forceinline__ float round_to(float x);
template <> __device__ __forceinline__ float round_to<float>(float x) { return x; }
template <> __device__ __forceinline__ float round_to<__nv_bfloat16>(float x) {
    return __bfloat162float(__float2bfloat16_rn(x));
}

// Counter-based Philox4x32-10 (Salmon et al., SC'11): 128 random bits per (counter c, key k0:k1), no state to carry
// between launches.  Used by the salt-and-pepper noise (augment.cu) and the Dropout3d keep factors (dropout.cu).
__device__ __forceinline__ void philox4x32_10(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
        const uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
        c[0] = n0, c[1] = lo1, c[2] = n2, c[3] = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---------------------------------------------------------------- virtual-craniectomy inside tests
// (transforms.py:286-296, utilities.py:127-178), shared by ctu_flap_mask_u8 (misc.cu) and the craniectomy encoder
// (augment.cu).  Sphere (shape 0) / box (shape 1) with an INTEGER radius r (np.random.randint, transforms.py:268):
// squared integer offsets are exact in I and sqrt is monotone, so np.linalg.norm(ord=2) <= r <=> dz^2 + dy^2 + dx^2 <= r^2
// bit for bit; r < 0 leaves nothing inside.  I = int while every squared distance fits 31 bits.
template <typename I>
__device__ __forceinline__ bool ball_inside(int shape, I dz, I dy, I dx, I r) {
    if (shape == 0) return r >= 0 && dz * dz + dy * dy + dx * dx <= r * r;
    return (dz < 0 ? -dz : dz) <= r && (dy < 0 ? -dy : dy) <= r && (dx < 0 ? -dx : dx) <= r;
}

// shape_3d(shape="flap") (utilities.py:145-166): the union of two cylinders along d (raster_geometry.cylinder, axis 0)
// and a cube (raster_geometry.cube).  raster_geometry is an un-vendored, unpinned dependency of the reference, so its
// published algorithm is RESTATED -- parity unpinned: relative positions become absolute grid origins
// x0 = rint((dim - 1) * rel) (round half to even), a cylinder is {(y-y0)^2 + (x-x0)^2 <= radius^2 and |z-z0| <= height/2},
// a cube is {|c - c0| <= side/2 on every axis}, all in float64 (the offsets are integers, so the sums are exact).
struct FlapHole {
    double z0, ey, ex1, ex2, qy, qx, half, r2;
};

__device__ __forceinline__ FlapHole flap_hole(int d, int h, int w, double c0, double c1, double c2, double size,
                                              double c_diam) {
    FlapHole f;
    // center_relative, z_edge_1, z_edge_2 (utilities.py:148-158) -> absolute origins
    f.z0 = rint((d - 1) * (c0 / d));
    f.ey = rint((h - 1) * ((c1 - size / 2) / h));
    f.ex1 = rint((w - 1) * ((c2 - size / 2) / w));
    f.ex2 = rint((w - 1) * ((c2 + size / 2) / w));
    f.qy = rint((h - 1) * (c1 / h));
    f.qx = rint((w - 1) * (c2 / w));
    f.half = size / 2;
    f.r2 = c_diam * c_diam;
    return f;
}

__device__ __forceinline__ bool flap_inside(const FlapHole& f, double z, double y, double x) {
    const bool in_height = fabs(z - f.z0) <= f.half;
    const double dy = y - f.ey, dy2 = dy * dy;
    return in_height && ((dy2 + (x - f.ex1) * (x - f.ex1) <= f.r2) || (dy2 + (x - f.ex2) * (x - f.ex2) <= f.r2) ||
                         (fabs(y - f.qy) <= f.half && fabs(x - f.qx) <= f.half));
}

// ---------------------------------------------------------------- concatenated sources
struct SrcMap {
    int nsrc;
    int ch[CTU_MAX_SRC];      // real channels per source
    int choff[CTU_MAX_SRC];   // offset of the source's first channel in the concatenated input
    int cboff[CTU_MAX_SRC];   // offset of the source's first 8-channel block
    int cb_total;             // total blocks over all sources
    int c_total;              // total real channels
};

static inline int make_srcmap(SrcMap& m, int nsrc, const int* h_src_channels) {
    if (nsrc < 1 || nsrc > CTU_MAX_SRC) {
        set_error("nsrc=%d out of range", nsrc);
        return CTU_ERR_INVALID;
    }
    m.nsrc = nsrc;
    int co = 0, bo = 0;
    for (int i = 0; i < nsrc; ++i) {
        if (h_src_channels[i] < 1) {
            set_error("source %d has %d channels", i, h_src_channels[i]);
            return CTU_ERR_INVALID;
        }
        m.ch[i] = h_src_channels[i];
        m.choff[i] = co;
        m.cboff[i] = bo;
        co += h_src_channels[i];
        bo += (h_src_channels[i] + 7) / 8;
    }
    for (int i = nsrc; i < CTU_MAX_SRC; ++i) m.ch[i] = m.choff[i] = m.cboff[i] = 0;
    m.cb_total = bo;
    m.c_total = co;
    return CTU_OK;
}

// Dispatch on the storage dtype of blocked activations.
#define CTU_DISPATCH_DTYPE(dtype, ...)                                  \
    do {                                                                \
        if ((dtype) == CTU_F32) {                                       \
            using T = float;                                            \
            __VA_ARGS__;                                                \
        } else if ((dtype) == CTU_BF16) {                               \
            using T = __nv_bfloat16;                                    \
            __VA_ARGS__;                                                \
        } else {                                                        \
            ctu::set_error("unknown dtype %d", (int)(dtype));           \
            return CTU_ERR_INVALID;                                     \
        }                                                               \
    } while (0)

}  // namespace ctu
