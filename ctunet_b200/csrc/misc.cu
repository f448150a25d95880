// Integer / byte glue kernels: virtual-craniectomy masking and CT preprocessing.
//   random_blank_patch / shape_3d   ctunet/pytorch/transforms.py:241-300, ctunet/utilities.py:127-178
//   HU windowing, thresholding, resampling: no reference implementation (SURVEY.md section 8c);
//   oracle/unet_oracle.py defines the semantics these kernels are bit-compared against.
#include "common.cuh"

namespace ctu {

constexpr int kVoxPerBlock = 4096;

__global__ void count_blocks_kernel(const unsigned char* __restrict__ img, long long nvox,
                                    long long* __restrict__ block_counts, long long* __restrict__ total) {
    const long long base = (long long)blockIdx.x * kVoxPerBlock;
    int cnt = 0;
    if (base + kVoxPerBlock <= nvox && (reinterpret_cast<uintptr_t>(img) & 15u) == 0) {
        // 256 threads x one 16-byte load = the block's 4096 voxels
        const uint4 u = reinterpret_cast<const uint4*>(img + base)[threadIdx.x];
        const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
        for (int j = 0; j < 4; ++j)      // a byte is non-zero <=> its low 7 bits carry into bit 7, or bit 7 is set
            cnt += __popc((((w[j] & 0x7f7f7f7fu) + 0x7f7f7f7fu) | w[j]) & 0x80808080u);
    } else {
        for (int i = threadIdx.x; i < kVoxPerBlock; i += blockDim.x) {
            long long v = base + i;
            if (v < nvox && img[v] > 0) ++cnt;
        }
    }
    __shared__ int red[8];
    int s = cnt;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        long long t = 0;
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += red[i];
        if (block_counts) block_counts[blockIdx.x] = t;
        if (total && t) atomicAdd((unsigned long long*)total, (unsigned long long)t);
    }
}

// np.argwhere(img > 0)[k] in C order: a block-wide prefix over the per-block counts finds the 4096-voxel block, a second
// prefix over its voxels (4 per thread) finds the voxel.  One block of 1024 threads.
__device__ __forceinline__ long long block_exclusive_scan(long long v, long long* warp_tot, long long& total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    long long inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const long long t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    __syncthreads();                      // warp_tot may still be read from a previous scan
    if (lane == 31) warp_tot[wid] = inc;
    __syncthreads();
    long long off = 0;
    total = 0;
    for (int i = 0; i < 32; ++i) {
        const long long t = warp_tot[i];
        if (i < wid) off += t;
        total += t;
    }
    return off + inc - v;
}

__global__ void __launch_bounds__(1024) kth_nonzero_kernel(const unsigned char* __restrict__ img, int d, int h, int w,
                                                           long long k, const long long* __restrict__ block_counts,
                                                           int nblocks, int* __restrict__ coords) {
    __shared__ long long warp_tot[32];
    __shared__ long long sel[2];          // chosen block, rank of the voxel inside it
    const long long nvox = (long long)d * h * w;
    if (threadIdx.x < 3) coords[threadIdx.x] = -1;
    if (threadIdx.x == 0) sel[0] = -1;
    // phase 1: every thread owns a contiguous chunk of the per-block counts
    const int per = (nblocks + 1023) / 1024;
    const int b0 = threadIdx.x * per, b1 = min(nblocks, b0 + per);
    long long mine = 0;
    for (int b = b0; b < b1; ++b) mine += block_counts[b];
    long long total;
    const long long before = block_exclusive_scan(mine, warp_tot, total);
    if (k >= total) return;               // fewer than k+1 non-zero voxels: coords stay -1 (uniform exit)
    if (k >= before && k < before + mine) {
        long long seen = before;
        for (int b = b0; b < b1; ++b) {
            if (seen + block_counts[b] > k) {
                sel[0] = b;
                sel[1] = k - seen;
                break;
            }
            seen += block_counts[b];
        }
    }
    __syncthreads();
    const long long blk = sel[0], rank = sel[1];
    // phase 2: 4096 voxels of the block, 4 consecutive voxels per thread
    const long long v0 = blk * kVoxPerBlock + 4LL * threadIdx.x;
    int nz[4], cnt = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        nz[j] = (v0 + j < nvox && img[v0 + j] > 0) ? 1 : 0;
        cnt += nz[j];
    }
    long long tot2;
    long long seen = block_exclusive_scan(cnt, warp_tot, tot2);
    if (rank >= seen && rank < seen + cnt) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (nz[j]) {
                if (seen == rank) {
                    const long long v = v0 + j;
                    coords[2] = (int)(v % w);
                    coords[1] = (int)((v / w) % h);
                    coords[0] = (int)(v / ((long long)w * h));
                }
                ++seen;
            }
        }
    }
}

__global__ void flap_mask_kernel(const unsigned char* __restrict__ img, unsigned char* __restrict__ masked,
                                 unsigned char* __restrict__ extracted, int d, int h, int w,
                                 const int* __restrict__ center, double size, int shape, long long nvox) {
    const long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= nvox) return;
    const int x = (int)(v % w);
    const int y = (int)((v / w) % h);
    const int z = (int)(v / ((long long)w * h));
    const double dz = (double)(z - center[0]), dy = (double)(y - center[1]), dx = (double)(x - center[2]);
    double dist;
    if (shape == 0) dist = sqrt(dz * dz + dy * dy + dx * dx);          // np.linalg.norm(ord=2), float64
    else dist = fmax(fabs(dz), fmax(fabs(dy), fabs(dx)));              // ord=inf
    const bool inside = dist <= size;                                   // utilities.py:177
    const bool on = img[v] != 0;
    masked[v] = (on && !inside) ? 1 : 0;                                // transforms.py:287
    extracted[v] = (on && inside) ? 1 : 0;                              // transforms.py:294
}

// shape_3d(shape="flap") (utilities.py:145-166): flap_hole / flap_inside (common.cuh)
__global__ void flap_shape_mask_kernel(const unsigned char* __restrict__ img, unsigned char* __restrict__ masked,
                                       unsigned char* __restrict__ extracted, int d, int h, int w,
                                       const int* __restrict__ center, double size, double c_diam, long long nvox) {
    const long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= nvox) return;
    const int x = (int)(v % w);
    const int y = (int)((v / w) % h);
    const int z = (int)(v / ((long long)w * h));
    const FlapHole f = flap_hole(d, h, w, (double)center[0], (double)center[1], (double)center[2], size, c_diam);
    const bool inside = flap_inside(f, z, y, x);                        // mask; shape_np = 1 - mask (utilities.py:165-166)
    const bool on = img[v] != 0;
    masked[v] = (on && !inside) ? 1 : 0;
    extracted[v] = (on && inside) ? 1 : 0;
}

// datasets.py:195-235 on the device: image channel 0 = the broken skull as float, channel 1 = the atlas
// (load_atlas_and_append_at_axis, datasets.py:30-47); targets = one_hot(label, 2) as float32 (datasets.py:209-214).
// 16 voxels per thread: one 16-byte load per mask, 16-byte stores.
__global__ void encode_flaprec_kernel(const unsigned char* __restrict__ broken, const unsigned char* __restrict__ full,
                                      const unsigned char* __restrict__ flap, const float* __restrict__ atlas,
                                      float* __restrict__ image, float* __restrict__ skull_t, float* __restrict__ flap_t,
                                      int cin, long long spatial) {
    const int b = blockIdx.y;
    const long long v0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 16;
    if (v0 >= spatial) return;
    const bool tg = skull_t != nullptr;       // image only: the fused head + loss kernels read the uint8 masks themselves
    const uint4 zero = make_uint4(0, 0, 0, 0);
    const uint4 ub = *reinterpret_cast<const uint4*>(broken + b * spatial + v0);
    const uint4 uf = tg ? *reinterpret_cast<const uint4*>(full + b * spatial + v0) : zero;
    const uint4 ul = tg ? *reinterpret_cast<const uint4*>(flap + b * spatial + v0) : zero;
    const uint32_t wb[4] = {ub.x, ub.y, ub.z, ub.w}, wf[4] = {uf.x, uf.y, uf.z, uf.w}, wl[4] = {ul.x, ul.y, ul.z, ul.w};
    float* img0 = image + (long long)b * cin * spatial + v0;
    float* sk0 = skull_t + (long long)b * 2 * spatial + v0;
    float* fl0 = flap_t + (long long)b * 2 * spatial + v0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        float vb[4], vf[4], vl[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            vb[j] = (float)((wb[i] >> (8 * j)) & 0xffu);                 // tensor.float(): the value itself
            vf[j] = ((wf[i] >> (8 * j)) & 0xffu) ? 1.f : 0.f;            // one_hot class of a {0,1} label
            vl[j] = ((wl[i] >> (8 * j)) & 0xffu) ? 1.f : 0.f;
        }
        *reinterpret_cast<float4*>(img0 + 4 * i) = make_float4(vb[0], vb[1], vb[2], vb[3]);
        if (tg) {
            *reinterpret_cast<float4*>(sk0 + 4 * i) = make_float4(1.f - vf[0], 1.f - vf[1], 1.f - vf[2], 1.f - vf[3]);
            *reinterpret_cast<float4*>(sk0 + spatial + 4 * i) = make_float4(vf[0], vf[1], vf[2], vf[3]);
            *reinterpret_cast<float4*>(fl0 + 4 * i) = make_float4(1.f - vl[0], 1.f - vl[1], 1.f - vl[2], 1.f - vl[3]);
            *reinterpret_cast<float4*>(fl0 + spatial + 4 * i) = make_float4(vl[0], vl[1], vl[2], vl[3]);
        }
        if (cin > 1) *reinterpret_cast<float4*>(img0 + spatial + 4 * i) = *reinterpret_cast<const float4*>(atlas + v0 + 4 * i);
    }
}

// The same encoding from BIT-PACKED masks (1 bit per voxel, voxel v = bit v & 7 of byte v >> 3, i.e. numpy's
// packbits(bitorder="little")): binary volumes cross PCIe at 3 bits per voxel instead of 24 bytes (float batch) or 3 bytes
// (uint8 masks).  Writes the float image (+ atlas channel) and, for the fused head + loss kernels, the two uint8 label masks.
// 16 voxels per thread: one 16-bit load per mask, four 16-byte image stores, one 16-byte store per label mask.
__global__ void encode_flaprec_bits_kernel(const unsigned char* __restrict__ broken, const unsigned char* __restrict__ full,
                                           const unsigned char* __restrict__ flap, const float* __restrict__ atlas,
                                           float* __restrict__ image, unsigned char* __restrict__ full_m,
                                           unsigned char* __restrict__ flap_m, int cin, long long spatial) {
    const int b = blockIdx.y;
    const long long v0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 16;
    if (v0 >= spatial) return;
    const long long byte0 = ((long long)b * spatial + v0) >> 3;
    const unsigned int wb = *reinterpret_cast<const unsigned short*>(broken + byte0);
    float* img0 = image + (long long)b * cin * spatial + v0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        *reinterpret_cast<float4*>(img0 + 4 * i) = make_float4((float)((wb >> (4 * i)) & 1u), (float)((wb >> (4 * i + 1)) & 1u),
                                                               (float)((wb >> (4 * i + 2)) & 1u), (float)((wb >> (4 * i + 3)) & 1u));
        if (cin > 1) *reinterpret_cast<float4*>(img0 + spatial + 4 * i) = *reinterpret_cast<const float4*>(atlas + v0 + 4 * i);
    }
    if (full_m != nullptr) {
        const unsigned int wf = *reinterpret_cast<const unsigned short*>(full + byte0);
        const unsigned int wl = *reinterpret_cast<const unsigned short*>(flap + byte0);
        uint32_t of[4], ol[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            of[i] = ((wf >> (4 * i)) & 1u) | (((wf >> (4 * i + 1)) & 1u) << 8) | (((wf >> (4 * i + 2)) & 1u) << 16) |
                    (((wf >> (4 * i + 3)) & 1u) << 24);
            ol[i] = ((wl >> (4 * i)) & 1u) | (((wl >> (4 * i + 1)) & 1u) << 8) | (((wl >> (4 * i + 2)) & 1u) << 16) |
                    (((wl >> (4 * i + 3)) & 1u) << 24);
        }
        *reinterpret_cast<uint4*>(full_m + (long long)b * spatial + v0) = make_uint4(of[0], of[1], of[2], of[3]);
        *reinterpret_cast<uint4*>(flap_m + (long long)b * spatial + v0) = make_uint4(ol[0], ol[1], ol[2], ol[3]);
    }
}

__global__ void hu_window_kernel(const short* __restrict__ hu, float* __restrict__ out, long long nvox, float lo,
                                 float hi) {
    const long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= nvox) return;
    float x = (float)hu[v];
    x = fminf(fmaxf(x, lo), hi);
    out[v] = __fdiv_rn(__fsub_rn(x, lo), __fsub_rn(hi, lo));
}

__global__ void hu_threshold_kernel(const short* __restrict__ hu, unsigned char* __restrict__ out, long long nvox,
                                    int thr) {
    const long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= nvox) return;
    out[v] = hu[v] >= thr ? 1 : 0;
}

// ---- 16-byte vector variants (the byte-per-thread kernels above reach 4-25 % of the HBM roofline: too few bytes in
// flight per thread).  The host uses them for the 16-aligned bulk of a volume and the scalar kernels for the tail.
__global__ void hu_window_vec_kernel(const short* __restrict__ hu, float* __restrict__ out, long long ngroups, float lo,
                                     float hi) {   // 16 voxels per thread: two 16-byte loads, four 16-byte stores
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ngroups) return;
    const uint4 a = reinterpret_cast<const uint4*>(hu)[2 * i], b = reinterpret_cast<const uint4*>(hu)[2 * i + 1];
    const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    const float den = __fsub_rn(hi, lo);
    float o[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const short sv = (short)((w[j >> 1] >> (16 * (j & 1))) & 0xffffu);
        float x = (float)sv;
        x = fminf(fmaxf(x, lo), hi);
        o[j] = __fdiv_rn(__fsub_rn(x, lo), den);
    }
    float4* dst = reinterpret_cast<float4*>(out) + 4 * i;
#pragma unroll
    for (int j = 0; j < 4; ++j) dst[j] = make_float4(o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
}

__global__ void hu_threshold_vec_kernel(const short* __restrict__ hu, unsigned char* __restrict__ out, long long ngroups,
                                        int thr) {   // 16 voxels per thread
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ngroups) return;
    const uint4 a = reinterpret_cast<const uint4*>(hu)[2 * i], b = reinterpret_cast<const uint4*>(hu)[2 * i + 1];
    const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    uint32_t o[4] = {0, 0, 0, 0};
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const short sv = (short)((w[j >> 1] >> (16 * (j & 1))) & 0xffffu);
        if ((int)sv >= thr) o[j >> 2] |= 1u << (8 * (j & 3));
    }
    reinterpret_cast<uint4*>(out)[i] = make_uint4(o[0], o[1], o[2], o[3]);
}

// sphere / box with an INTEGER radius (ball_inside, common.cuh); 16 voxels of one row per thread
template <typename I>   // I = int when every squared distance fits 31 bits (volumes up to 16384 voxels a side), else long long
__global__ void flap_mask_vec_kernel(const unsigned char* __restrict__ img, unsigned char* __restrict__ masked,
                                     unsigned char* __restrict__ extracted, int d, int h, int w, const int* __restrict__ center,
                                     long long size_ll, int shape, long long ngroups) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ngroups) return;
    const int wg = w >> 4;
    const int x0 = (int)(i % wg) << 4;
    const int y = (int)((i / wg) % h);
    const int z = (int)(i / ((long long)wg * h));
    const I size = (I)size_ll;
    const I dz = z - center[0], dy = y - center[1], cx = center[2];
    const uint4 u = reinterpret_cast<const uint4*>(img)[i];
    const uint32_t wv[4] = {u.x, u.y, u.z, u.w};
    uint32_t m[4] = {0, 0, 0, 0}, e[4] = {0, 0, 0, 0};
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const bool inside = ball_inside<I>(shape, dz, dy, x0 + j - cx, size);
        const bool on = ((wv[j >> 2] >> (8 * (j & 3))) & 0xffu) != 0;
        if (on && !inside) m[j >> 2] |= 1u << (8 * (j & 3));
        if (on && inside) e[j >> 2] |= 1u << (8 * (j & 3));
    }
    reinterpret_cast<uint4*>(masked)[i] = make_uint4(m[0], m[1], m[2], m[3]);
    reinterpret_cast<uint4*>(extracted)[i] = make_uint4(e[0], e[1], e[2], e[3]);
}

// the flap shape, 16 voxels of one row per thread (flap_hole / flap_inside, common.cuh)
__global__ void flap_shape_mask_vec_kernel(const unsigned char* __restrict__ img, unsigned char* __restrict__ masked,
                                           unsigned char* __restrict__ extracted, int d, int h, int w,
                                           const int* __restrict__ center, double size, double c_diam, long long ngroups) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ngroups) return;
    const int wg = w >> 4;
    const int x0 = (int)(i % wg) << 4;
    const int y = (int)((i / wg) % h);
    const int z = (int)(i / ((long long)wg * h));
    const FlapHole f = flap_hole(d, h, w, (double)center[0], (double)center[1], (double)center[2], size, c_diam);
    const uint4 u = reinterpret_cast<const uint4*>(img)[i];
    const uint32_t wv[4] = {u.x, u.y, u.z, u.w};
    uint32_t m[4] = {0, 0, 0, 0}, e[4] = {0, 0, 0, 0};
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const bool inside = flap_inside(f, z, y, x0 + j);
        const bool on = ((wv[j >> 2] >> (8 * (j & 3))) & 0xffu) != 0;
        if (on && !inside) m[j >> 2] |= 1u << (8 * (j & 3));
        if (on && inside) e[j >> 2] |= 1u << (8 * (j & 3));
    }
    reinterpret_cast<uint4*>(masked)[i] = make_uint4(m[0], m[1], m[2], m[3]);
    reinterpret_cast<uint4*>(extracted)[i] = make_uint4(e[0], e[1], e[2], e[3]);
}

__device__ __forceinline__ int nearest_src(int dst, int in_size, float scale) {
    int i = (int)floorf(__fmul_rn((float)dst, scale));
    return i < in_size - 1 ? i : in_size - 1;
}

template <typename V>
__global__ void resample_nearest_kernel(const V* __restrict__ src, V* __restrict__ dst, int sd, int sh, int sw, int dd,
                                        int dh, int dw, float fz, float fy, float fx, long long total) {
    const long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= total) return;
    const int x = (int)(v % dw);
    const int y = (int)((v / dw) % dh);
    const int z = (int)(v / ((long long)dw * dh));
    const int iz = nearest_src(z, sd, fz), iy = nearest_src(y, sh, fy), ix = nearest_src(x, sw, fx);
    dst[v] = src[((long long)iz * sh + iy) * sw + ix];
}

__global__ void nearest_index_kernel(int* __restrict__ idx, int out_size, int in_size, float scale) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < out_size) idx[i] = nearest_src(i, in_size, scale);
}

// F.interpolate(mode='trilinear', align_corners=False): src = scale*(dst+0.5)-0.5 clamped at 0
__device__ __forceinline__ void lin_coord(int dst, int in_size, float scale, int& i0, int& i1, float& l0, float& l1) {
    float s = __fsub_rn(__fmul_rn(scale, __fadd_rn((float)dst, 0.5f)), 0.5f);
    if (s < 0.f) s = 0.f;
    i0 = (int)s;
    if (i0 > in_size - 1) i0 = in_size - 1;
    i1 = i0 + (i0 < in_size - 1 ? 1 : 0);
    l1 = __fsub_rn(s, (float)i0);
    l0 = __fsub_rn(1.f, l1);
}

__global__ void resample_trilinear_kernel(const float* __restrict__ src, float* __restrict__ dst, int sd, int sh, int sw,
                                          int dd, int dh, int dw, float fz, float fy, float fx, long long total) {
    const long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= total) return;
    const int x = (int)(v % dw);
    const int y = (int)((v / dw) % dh);
    const int z = (int)(v / ((long long)dw * dh));
    int z0, z1, y0, y1, x0, x1;
    float lz0, lz1, ly0, ly1, lx0, lx1;
    lin_coord(z, sd, fz, z0, z1, lz0, lz1);
    lin_coord(y, sh, fy, y0, y1, ly0, ly1);
    lin_coord(x, sw, fx, x0, x1, lx0, lx1);
    auto at = [&](int zz, int yy, int xx) { return __ldg(src + ((long long)zz * sh + yy) * sw + xx); };
    const float a = ly0 * (lx0 * at(z0, y0, x0) + lx1 * at(z0, y0, x1)) + ly1 * (lx0 * at(z0, y1, x0) + lx1 * at(z0, y1, x1));
    const float b = ly0 * (lx0 * at(z1, y0, x0) + lx1 * at(z1, y0, x1)) + ly1 * (lx0 * at(z1, y1, x0) + lx1 * at(z1, y1, x1));
    dst[v] = lz0 * a + lz1 * b;
}

}  // namespace ctu

using namespace ctu;

static inline bool aligned16_host(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

extern "C" {

int ctu_count_nonzero_u8(const unsigned char* img, long long nvox, long long* count, ctu_stream stream) {
    CTU_REQUIRE(img && count && nvox > 0, "ctu_count_nonzero_u8: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(count, 0, sizeof(long long), st);
    if (e != cudaSuccess) {
        set_error("ctu_count_nonzero_u8: memset: %s", cudaGetErrorString(e));
        return (int)e;
    }
    count_blocks_kernel<<<cdiv(nvox, kVoxPerBlock), 256, 0, st>>>(img, nvox, nullptr, count);
    return check_launch("ctu_count_nonzero_u8");
}

int ctu_kth_nonzero_u8(const unsigned char* img, int d, int h, int w, long long k, long long* block_counts, int* coords,
                       ctu_stream stream) {
    CTU_REQUIRE(img && block_counts && coords && d > 0 && h > 0 && w > 0 && k >= 0, "ctu_kth_nonzero_u8: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    const long long nvox = (long long)d * h * w;
    const int nblocks = cdiv(nvox, kVoxPerBlock);
    count_blocks_kernel<<<nblocks, 256, 0, st>>>(img, nvox, block_counts, nullptr);
    kth_nonzero_kernel<<<1, 1024, 0, st>>>(img, d, h, w, k, block_counts, nblocks, coords);
    return check_launch("ctu_kth_nonzero_u8");
}

int ctu_flap_mask_u8(const unsigned char* img, unsigned char* masked, unsigned char* extracted, int d, int h, int w,
                     const int* center, double size, int shape, double c_diam, ctu_stream stream) {
    CTU_REQUIRE(img && masked && extracted && center && d > 0 && h > 0 && w > 0 && shape >= 0 && shape <= 2,
                "ctu_flap_mask_u8: bad arguments (shape 0 sphere / 1 box / 2 flap)");
    const long long nvox = (long long)d * h * w;
    cudaStream_t st = (cudaStream_t)stream;
    const bool vec = (w % 16 == 0) && aligned16_host(img) && aligned16_host(masked) && aligned16_host(extracted);
    const long long ngroups = nvox / 16;
    if (shape == 2) {
        if (vec) flap_shape_mask_vec_kernel<<<cdiv(ngroups, 256), 256, 0, st>>>(img, masked, extracted, d, h, w, center, size, c_diam, ngroups);
        else flap_shape_mask_kernel<<<cdiv(nvox, 256), 256, 0, st>>>(img, masked, extracted, d, h, w, center, size, c_diam, nvox);
    } else if (vec && size >= 0 && size < 1048576.0 && size == (double)(long long)size) {
        // int32: 3 * 16384^2 < 2^31; a radius beyond the volume diagonal is clamped (everything is inside either way)
        if (d <= 16384 && h <= 16384 && w <= 16384)
            flap_mask_vec_kernel<int><<<cdiv(ngroups, 256), 256, 0, st>>>(img, masked, extracted, d, h, w, center,
                                                                         size > 28378.0 ? 28378LL : (long long)size, shape, ngroups);
        else
            flap_mask_vec_kernel<long long><<<cdiv(ngroups, 256), 256, 0, st>>>(img, masked, extracted, d, h, w, center, (long long)size, shape, ngroups);
    } else {
        flap_mask_kernel<<<cdiv(nvox, 256), 256, 0, st>>>(img, masked, extracted, d, h, w, center, size, shape, nvox);
    }
    return check_launch("ctu_flap_mask_u8");
}

int ctu_encode_flaprec_u8(const unsigned char* broken, const unsigned char* full, const unsigned char* flap,
                          const float* atlas, float* image, float* skull_target, float* flap_target, int batch,
                          int in_channels, long long spatial, ctu_stream stream) {
    CTU_REQUIRE(broken && image && batch > 0 && spatial > 0, "ctu_encode_flaprec_u8: bad arguments");
    CTU_REQUIRE((skull_target != nullptr) == (flap_target != nullptr) && (skull_target == nullptr || (full && flap)),
                "ctu_encode_flaprec_u8: both targets (with both label masks) or neither");
    CTU_REQUIRE(in_channels == 1 || (in_channels == 2 && atlas), "ctu_encode_flaprec_u8: 1 input channel, or 2 with an atlas");
    CTU_REQUIRE(spatial % 16 == 0, "ctu_encode_flaprec_u8: the volume size must be a multiple of 16 voxels");
    dim3 grid(cdiv(spatial / 16, 256), batch);
    encode_flaprec_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(broken, full, flap, atlas, image, skull_target, flap_target,
                                                                  in_channels, spatial);
    return check_launch("ctu_encode_flaprec_u8");
}

int ctu_encode_flaprec_bits(const unsigned char* broken_bits, const unsigned char* full_bits, const unsigned char* flap_bits,
                            const float* atlas, float* image, unsigned char* full_mask, unsigned char* flap_mask, int batch,
                            int in_channels, long long spatial, ctu_stream stream) {
    CTU_REQUIRE(broken_bits && image && batch > 0 && spatial > 0, "ctu_encode_flaprec_bits: bad arguments");
    CTU_REQUIRE((full_mask != nullptr) == (flap_mask != nullptr) && (full_mask == nullptr || (full_bits && flap_bits)),
                "ctu_encode_flaprec_bits: both label masks (with both bit volumes) or neither");
    CTU_REQUIRE(in_channels == 1 || (in_channels == 2 && atlas), "ctu_encode_flaprec_bits: 1 input channel, or 2 with an atlas");
    CTU_REQUIRE(spatial % 16 == 0, "ctu_encode_flaprec_bits: the volume size must be a multiple of 16 voxels");
    dim3 grid(cdiv(spatial / 16, 256), batch);
    encode_flaprec_bits_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(broken_bits, full_bits, flap_bits, atlas, image, full_mask,
                                                                       flap_mask, in_channels, spatial);
    return check_launch("ctu_encode_flaprec_bits");
}

int ctu_hu_window(const short* hu, float* out, long long nvox, float lo, float hi, ctu_stream stream) {
    CTU_REQUIRE(hu && out && nvox > 0 && hi > lo, "ctu_hu_window: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    long long done = 0;
    if (aligned16_host(hu) && aligned16_host(out) && nvox >= 16) {
        const long long ngroups = nvox / 16;
        hu_window_vec_kernel<<<cdiv(ngroups, 256), 256, 0, st>>>(hu, out, ngroups, lo, hi);
        done = ngroups * 16;
    }
    if (done < nvox) hu_window_kernel<<<cdiv(nvox - done, 256), 256, 0, st>>>(hu + done, out + done, nvox - done, lo, hi);
    return check_launch("ctu_hu_window");
}

int ctu_hu_threshold(const short* hu, unsigned char* out, long long nvox, int thr, ctu_stream stream) {
    CTU_REQUIRE(hu && out && nvox > 0, "ctu_hu_threshold: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    long long done = 0;
    if (aligned16_host(hu) && aligned16_host(out) && nvox >= 16) {
        const long long ngroups = nvox / 16;
        hu_threshold_vec_kernel<<<cdiv(ngroups, 256), 256, 0, st>>>(hu, out, ngroups, thr);
        done = ngroups * 16;
    }
    if (done < nvox) hu_threshold_kernel<<<cdiv(nvox - done, 256), 256, 0, st>>>(hu + done, out + done, nvox - done, thr);
    return check_launch("ctu_hu_threshold");
}

static inline float nscale(int in_size, int out_size) { return (float)in_size / (float)out_size; }

int ctu_resample_nearest_f32(const float* src, float* dst, int sd, int sh, int sw, int dd, int dh, int dw,
                             ctu_stream stream) {
    CTU_REQUIRE(src && dst && sd > 0 && sh > 0 && sw > 0 && dd > 0 && dh > 0 && dw > 0, "ctu_resample_nearest_f32: bad arguments");
    const long long total = (long long)dd * dh * dw;
    resample_nearest_kernel<float><<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(src, dst, sd, sh, sw, dd, dh, dw, nscale(sd, dd), nscale(sh, dh), nscale(sw, dw), total);
    return check_launch("ctu_resample_nearest_f32");
}

int ctu_resample_nearest_u8(const unsigned char* src, unsigned char* dst, int sd, int sh, int sw, int dd, int dh, int dw,
                            ctu_stream stream) {
    CTU_REQUIRE(src && dst && sd > 0 && sh > 0 && sw > 0 && dd > 0 && dh > 0 && dw > 0, "ctu_resample_nearest_u8: bad arguments");
    const long long total = (long long)dd * dh * dw;
    resample_nearest_kernel<unsigned char><<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(src, dst, sd, sh, sw, dd, dh, dw, nscale(sd, dd), nscale(sh, dh), nscale(sw, dw), total);
    return check_launch("ctu_resample_nearest_u8");
}

int ctu_resample_nearest_index(int* idx, int out_size, int in_size, ctu_stream stream) {
    CTU_REQUIRE(idx && out_size > 0 && in_size > 0, "ctu_resample_nearest_index: bad arguments");
    nearest_index_kernel<<<cdiv(out_size, 256), 256, 0, (cudaStream_t)stream>>>(idx, out_size, in_size, nscale(in_size, out_size));
    return check_launch("ctu_resample_nearest_index");
}

int ctu_resample_trilinear_f32(const float* src, float* dst, int sd, int sh, int sw, int dd, int dh, int dw,
                               ctu_stream stream) {
    CTU_REQUIRE(src && dst && sd > 0 && sh > 0 && sw > 0 && dd > 0 && dh > 0 && dw > 0, "ctu_resample_trilinear_f32: bad arguments");
    const long long total = (long long)dd * dh * dw;
    resample_trilinear_kernel<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(src, dst, sd, sh, sw, dd, dh, dw, nscale(sd, dd), nscale(sh, dh), nscale(sw, dw), total);
    return check_launch("ctu_resample_trilinear_f32");
}

}  // extern "C"
