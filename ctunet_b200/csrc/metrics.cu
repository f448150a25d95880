// Reporting metrics of the loss handlers on the device: hard-label Dice coefficient and Hausdorff distance.
//   utils.dice_coeff   ctunet/utilities.py:53-60   (monai.metrics.compute_meandice on one_hot(argmax(pred)))
//   utils.hausdorff    ctunet/utilities.py:63-70   (monai.metrics.compute_hausdorff_distance, nan/inf -> max(shape))
//   call sites         ctunet/pytorch/ProblemHandler.py:84-88, 277-295  (every stock .ini switches them on)
// monai is an undeclared, unpinned dependency of the reference (not installable here): its published algorithm is
// restated (oracle/ref_stubs/monai/metrics.py is the CPU statement the tests compare with) -> PARITY UNPINNED.
//
// Hausdorff = integer work: edge voxels (mask minus its 6-neighbourhood erosion, outside = background), an EXACT squared
// Euclidean distance transform to the other surface (three separable min-plus passes over int32 squared distances), a max
// over the edge voxels, one sqrt in double at the end.  All HBM/L2-resident byte and int32 traffic; nothing syncs.
//
// Surface metrics (utilities.surface_metrics, DESIGN.md section 7d; oracle tests/surface_oracle.py) run on the same edge
// kernel and EDT: the EDT in int32 (voxel units) or in double with per-axis weights s^2 (spacing), a last pass that
// reduces max / count <= tolerance / per-CTA sums and lists the keys, a radix select for the percentile's order
// statistics, and a finalize that restates numpy's linear percentile.
#include <cooperative_groups.h>

#include "common.cuh"

namespace ctu {

constexpr int kInfD2 = 1 << 29;
constexpr int kMetThreads = 256;

// ---------------------------------------------------------------- masks + Dice counts
// item = (b, cls-1): pmask = [argmax_c pred == cls], tmask = [target[cls] == 1]; counts[item] = {sum t*m, sum t, sum m}
template <int C>
__global__ void __launch_bounds__(kMetThreads) seg_masks_kernel(const float* __restrict__ pred, const float* __restrict__ target,
                                                                long long spatial, unsigned char* __restrict__ pmask,
                                                                unsigned char* __restrict__ tmask, double* __restrict__ counts) {
    const int b = blockIdx.y;
    const float* pb = pred + (long long)b * C * spatial;
    const float* tb = target + (long long)b * C * spatial;
    float inter[C - 1], ysum[C - 1];
    int psum[C - 1];
#pragma unroll
    for (int c = 0; c < C - 1; ++c) inter[c] = ysum[c] = 0.f, psum[c] = 0;
    for (long long v = (long long)blockIdx.x * kMetThreads + threadIdx.x; v < spatial; v += (long long)gridDim.x * kMetThreads) {
        int am = 0;
        float best = __ldg(pb + v);
#pragma unroll
        for (int c = 1; c < C; ++c) {
            const float x = __ldg(pb + c * spatial + v);
            if (x > best || (x != x && best == best)) best = x, am = c;       // torch.argmax: first max, NaN wins
        }
#pragma unroll
        for (int c = 1; c < C; ++c) {
            const float t = __ldg(tb + c * spatial + v);
            const int m = am == c;
            inter[c - 1] += m ? t : 0.f;
            ysum[c - 1] += t;
            psum[c - 1] += m;
            if (pmask) {
                pmask[((long long)b * (C - 1) + (c - 1)) * spatial + v] = (unsigned char)m;
                tmask[((long long)b * (C - 1) + (c - 1)) * spatial + v] = (unsigned char)(t == 1.0f);
            }
        }
    }
    __shared__ double red[kMetThreads / 32][3 * (C - 1)];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int c = 0; c < C - 1; ++c) {
        const double a = warp_sum((double)inter[c]), y = warp_sum((double)ysum[c]), p = warp_sum((double)psum[c]);
        if (lane == 0) red[wid][3 * c] = a, red[wid][3 * c + 1] = y, red[wid][3 * c + 2] = p;
    }
    __syncthreads();
    if (threadIdx.x < 3 * (C - 1)) {
        double s = 0;
        for (int w = 0; w < kMetThreads / 32; ++w) s += red[w][threadIdx.x];
        atomicAdd(counts + ((long long)b * (C - 1)) * 3 + threadIdx.x, s);
    }
}

__global__ void dice_coeff_finalize_kernel(const double* __restrict__ counts, int items, float* __restrict__ out) {
    // monai: f = 2*I / (y_o + y_pred_o) in float32, NaN where y_o == 0; the reference takes torch.mean over [B, C-1]
    float acc = 0.f;
    for (int i = 0; i < items; ++i) {
        const float I = (float)counts[3 * i], yo = (float)counts[3 * i + 1], po = (float)counts[3 * i + 2];
        acc += yo > 0.f ? (2.0f * I) / (yo + po) : __int_as_float(0x7fc00000);
    }
    out[0] = acc / (float)items;
}

// ---------------------------------------------------------------- edges, Dice and edge counts
// edge = mask AND NOT (all six face neighbours set); voxels outside the volume are background (scipy binary_erosion,
// border_value = 0).  A voxel is in a mask when it is non-zero (NaN counts, -0.0 does not).
__device__ __forceinline__ bool fg(unsigned char v) { return v != 0; }
__device__ __forceinline__ bool fg(float v) { return v != 0.0f; }

template <typename T>
__device__ __forceinline__ bool interior(const T* __restrict__ m, long long v, int x, int y, int z, int d, int h, int w) {
    const long long hw = (long long)w * h;
    return x > 0 && x < w - 1 && y > 0 && y < h - 1 && z > 0 && z < d - 1 && fg(m[v - 1]) && fg(m[v + 1]) && fg(m[v - w]) &&
           fg(m[v + w]) && fg(m[v - hw]) && fg(m[v + hw]);
}

// Pair p = blockIdx.y: prediction mask pred + p * pstride, target mask target + p * tstride.  Writes the edge flags of
// set 2p (prediction) and 2p + 1 (target), so that partner(set) = set ^ 1, and adds
// stats[5p + {0..4}] = {|P|, |T|, |P n T|, #edges(P), #edges(T)}: counted per thread, reduced per CTA, 5 atomics per CTA.
template <typename TP, typename TT>
__global__ void __launch_bounds__(kMetThreads) mask_edges_kernel(const TP* __restrict__ pred, long long pstride,
                                                                 const TT* __restrict__ target, long long tstride,
                                                                 unsigned char* __restrict__ edge, int d, int h, int w,
                                                                 unsigned long long* __restrict__ stats) {
    const long long spatial = (long long)d * h * w;
    const int pair = blockIdx.y;
    const TP* pm = pred + pair * pstride;
    const TT* tm = target + pair * tstride;
    unsigned char* pe = edge + 2LL * pair * spatial;
    unsigned char* te = pe + spatial;
    int c[5] = {0, 0, 0, 0, 0};
    for (long long v = (long long)blockIdx.x * kMetThreads + threadIdx.x; v < spatial; v += (long long)gridDim.x * kMetThreads) {
        const int x = (int)(v % w), y = (int)((v / w) % h), z = (int)(v / ((long long)w * h));
        const int a = fg(pm[v]), t = fg(tm[v]);
        const int ea = a && !interior(pm, v, x, y, z, d, h, w);
        const int et = t && !interior(tm, v, x, y, z, d, h, w);
        pe[v] = (unsigned char)ea;
        te[v] = (unsigned char)et;
        c[0] += a, c[1] += t, c[2] += a & t, c[3] += ea, c[4] += et;
    }
    __shared__ int red[kMetThreads / 32][5];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < 5; ++i) {
        const int s = __reduce_add_sync(0xffffffffu, c[i]);
        if (lane == 0) red[wid][i] = s;
    }
    __syncthreads();
    if (threadIdx.x < 5) {
        long long s = 0;
        for (int k = 0; k < kMetThreads / 32; ++k) s += red[k][threadIdx.x];
        if (s) atomicAdd(stats + 5LL * pair + threadIdx.x, (unsigned long long)s);
    }
}

// ---------------------------------------------------------------- distance types of the EDT
// int: squared distances in voxel units (exact; kInfD2 = no edge voxel); term(k) = k^2, the axis weight is unused.
// double: squared distances with per-axis weights s^2 (voxel spacing); term(k) = s^2 k^2; +inf = no edge voxel.
// key(): an unsigned integer with the order of the distances (int: the value; double: the bit pattern of a non-negative
// double), so that one radix select serves both.  A column tile of the min-plus passes is 128 bytes wide: 32 int lanes or
// 16 double lanes (a 1024-long double column of 32 lanes would be 256 KB, over the 227 KB a block can have).
template <typename T> struct Dist;
template <> struct Dist<int> {
    static constexpr int kLanes = 32;
    __device__ static __forceinline__ int inf() { return kInfD2; }
    __device__ static __forceinline__ int term(int k, int) { return k * k; }
    __device__ static __forceinline__ unsigned long long key(int d2) { return (unsigned long long)(unsigned)d2; }
};
template <> struct Dist<double> {
    static constexpr int kLanes = 16;
    __device__ static __forceinline__ double inf() { return __longlong_as_double(0x7ff0000000000000LL); }
    __device__ static __forceinline__ double term(int k, double s2) { return __dmul_rn(s2, (double)(k * k)); }
    __device__ static __forceinline__ unsigned long long key(double d2) { return (unsigned long long)__double_as_longlong(d2); }
};

// Euclidean distance of a key: sqrt in double, as scipy's distance_transform_edt takes it.
__device__ __forceinline__ double key_distance(unsigned long long key, bool weighted) {
    return __dsqrt_rn(weighted ? __longlong_as_double((long long)key) : (double)key);
}

// ---------------------------------------------------------------- squared EDT, pass 1 (along w)
// g[z][y][x] = min over edge voxels x' of the row of term(x - x'), inf if the row has none.
template <typename T>
__global__ void edt_row_kernel(const unsigned char* __restrict__ edge, T* __restrict__ g, int w, long long rows, T wx) {
    extern __shared__ unsigned char srow[];
    const int rpb = blockDim.y;
    const long long row = (long long)blockIdx.x * rpb + threadIdx.y;
    unsigned char* r = srow + threadIdx.y * w;
    if (row < rows)
        for (int x = threadIdx.x; x < w; x += blockDim.x) r[x] = edge[row * w + x];
    __syncthreads();
    if (row >= rows) return;
    for (int x = threadIdx.x; x < w; x += blockDim.x) {
        T best = Dist<T>::inf();
        // nearest set voxel left and right of x: walk outwards, stop at the first hit
        for (int k = 0; k < w; ++k) {
            const int a = x - k, b = x + k;
            if ((a >= 0 && r[a]) || (b < w && r[b])) {
                best = Dist<T>::term(k, wx);
                break;
            }
            if (a < 0 && b >= w) break;
        }
        g[row * w + x] = best;
    }
}

// ---------------------------------------------------------------- squared EDT, passes 2 and 3 (min-plus along L)
// Volume viewed as [outer][L][inner]: out[o][l][i] = min_l' (in[o][l'][i] + term(l - l')).  A block owns (o, a tile of
// kLanes inner positions): the whole column tile sits in shared memory.  The last pass reduces, instead of storing, over
// the voxels of the PARTNER edge set (set ^ 1), i.e. over the directed distances from the partner surface to this one:
//   kMax      max d2 into maxd2[set] (utilities.hausdorff);
//   kSurface  per set: max key, #{sqrt(d2) <= tau} and #keys into acc.cnt[3 set + {1, 2, 0}], the sum of sqrt(d2) per CTA
//             into acc.partial[set][blockIdx.x] (reduced later in a fixed order), and every key appended to acc.keys
//             (warp-aggregated slots: the order is not fixed, but only the order statistics of the list are used).
enum { kStore = 0, kMax = 1, kSurface = 2 };
struct SurfAcc {
    unsigned long long* keys;       // [set][set_stride]
    unsigned long long* cnt;        // [set][3]: #keys, max key, #{distance <= tau}
    double* partial;                // [set][gridDim.x]
    double tau;
};

template <typename T, int MODE>
__global__ void edt_axis_kernel(const T* __restrict__ in, T* __restrict__ out, int L, long long inner,
                                long long outer, long long set_stride, T wl, const unsigned char* __restrict__ edge,
                                int* __restrict__ maxd2, SurfAcc acc) {
    constexpr int LN = Dist<T>::kLanes;
    extern __shared__ __align__(16) unsigned char edt_smem[];
    T* col = reinterpret_cast<T*>(edt_smem);      // [L][LN]
    const int set = blockIdx.z;
    const long long tiles = (inner + LN - 1) / LN;
    const long long o = blockIdx.x / tiles;
    const long long i0 = (blockIdx.x % tiles) * LN;
    const long long base = (long long)set * set_stride + o * L * inner;
    const int lx = threadIdx.x;                    // inner lane
    const bool ok = i0 + lx < inner;
    for (int l = threadIdx.y; l < L; l += blockDim.y) col[l * LN + lx] = ok ? in[base + (long long)l * inner + i0 + lx] : Dist<T>::inf();
    __syncthreads();
    int local_max = -1;
    unsigned long long kmax = 0;
    double sum = 0.0;
    int le = 0;
    for (int l = threadIdx.y; l < L; l += blockDim.y) {
        T best = col[l * LN + lx];
        // candidates further away than sqrt(best) cannot win: shrink the window as best improves
        for (int k = 1; k < L; ++k) {
            const T kk = Dist<T>::term(k, wl);
            if (kk >= best) break;
            const int a = l - k, b = l + k;
            if (a >= 0) best = min(best, col[a * LN + lx] + kk);
            if (b < L) best = min(best, col[b * LN + lx] + kk);
            if (a < 0 && b >= L) break;
        }
        if (!ok) continue;
        const long long idx = o * L * inner + (long long)l * inner + i0 + lx;
        if constexpr (MODE == kMax) {
            const unsigned char* pe = edge + (long long)(set ^ 1) * set_stride;      // the partner set's edges
            if (pe[idx]) local_max = max(local_max, best);
        } else if constexpr (MODE == kSurface) {
            if (edge[(long long)(set ^ 1) * set_stride + idx]) {
                const unsigned long long key = Dist<T>::key(best);
                const double dist = key_distance(key, sizeof(T) == 8);
                kmax = max(kmax, key);
                sum += dist;
                le += dist <= acc.tau;
                cooperative_groups::coalesced_group g = cooperative_groups::coalesced_threads();
                unsigned long long slot = 0;
                if (g.thread_rank() == 0) slot = atomicAdd(acc.cnt + 3 * set, (unsigned long long)g.size());
                slot = g.shfl(slot, 0) + g.thread_rank();
                acc.keys[(long long)set * set_stride + slot] = key;
            }
        } else {
            out[(long long)set * set_stride + idx] = best;
        }
    }
    if constexpr (MODE == kMax) {
        for (int off = 16; off > 0; off >>= 1) local_max = max(local_max, __shfl_xor_sync(0xffffffffu, local_max, off));
        if (lx == 0 && local_max >= 0) atomicMax(maxd2 + set, local_max);
    } else if constexpr (MODE == kSurface) {
        __shared__ unsigned long long smax[8];
        __shared__ double ssum[8];
        __shared__ int sle[8];
        const int tid = threadIdx.y * LN + lx, lane = tid & 31, wid = tid >> 5;
        for (int off = 16; off > 0; off >>= 1) {
            kmax = max(kmax, __shfl_xor_sync(0xffffffffu, kmax, off));
            sum += __shfl_xor_sync(0xffffffffu, sum, off);
            le += __shfl_xor_sync(0xffffffffu, le, off);
        }
        if (lane == 0) smax[wid] = kmax, ssum[wid] = sum, sle[wid] = le;
        __syncthreads();
        if (tid == 0) {
            for (int k = 1; k < 8; ++k) kmax = max(kmax, smax[k]), sum += ssum[k], le += sle[k];
            acc.partial[(long long)set * gridDim.x + blockIdx.x] = sum;
            if (kmax) atomicMax(acc.cnt + 3 * set + 1, kmax);
            if (le) atomicAdd(acc.cnt + 3 * set + 2, (unsigned long long)le);
        }
    }
}

// sets come in pairs (2p = prediction, 2p+1 = target).  maxd2[2p] = max over target-edge voxels of d2 to the prediction
// surface, maxd2[2p+1] the other direction.  Empty surface on either side -> NaN / inf in monai -> inf_alt (utilities.py:69).
__global__ void hausdorff_finalize_kernel(const int* __restrict__ maxd2, const unsigned long long* __restrict__ stats,
                                          int pairs, double inf_alt, double* __restrict__ out) {
    double acc = 0;
    for (int p = 0; p < pairs; ++p) {
        double hd = inf_alt;
        if (stats[5 * p + 3] && stats[5 * p + 4]) hd = sqrt((double)max(maxd2[2 * p], maxd2[2 * p + 1]));
        acc += hd;
    }
    out[0] = acc / pairs;
}

// ---------------------------------------------------------------- percentile: exact order statistics by radix select
// numpy.percentile(x, p) (method "linear", numpy 2.3) restated operation by operation for n sorted values:
// q = p / 100, vi = (n - 1) q, prev = floor(vi), both indices = n - 1 and prev = -1 when vi >= n - 1; g = vi - prev.
__device__ __forceinline__ void pct_index(unsigned long long n, double percentile, unsigned long long& lo,
                                          unsigned long long& hi, double& g) {
    const double vi = __dmul_rn((double)(n - 1), __ddiv_rn(percentile, 100.0));
    double prev = floor(vi);
    if (vi >= (double)(n - 1)) {
        lo = hi = n - 1;
        prev = -1.0;
    } else {
        lo = (unsigned long long)prev;
        hi = lo + 1;
    }
    g = __dsub_rn(vi, prev);
}

// numpy's _lerp: a + (b - a) g, or b - (b - a)(1 - g) where g >= 0.5; no FMA contraction.
__device__ __forceinline__ double np_lerp(double a, double b, double g) {
    const double diff = __dsub_rn(b, a);
    return g >= 0.5 ? __dsub_rn(b, __dmul_rn(diff, __dsub_rn(1.0, g))) : __dadd_rn(a, __dmul_rn(diff, g));
}

// sel[2 item + {0, 1}] = {key prefix found so far, rank left inside it}, item = 2 set + {0: lower, 1: upper index}.
__global__ void pct_rank_kernel(const unsigned long long* __restrict__ cnt, int sets, double percentile,
                                unsigned long long* __restrict__ sel) {
    for (int item = blockIdx.x * blockDim.x + threadIdx.x; item < 2 * sets; item += gridDim.x * blockDim.x) {
        const unsigned long long n = cnt[3 * (item >> 1)];
        unsigned long long lo = 0, hi = 0;
        double g;
        if (n) pct_index(n, percentile, lo, hi, g);
        sel[2 * item] = 0;
        sel[2 * item + 1] = (item & 1) ? hi : lo;
    }
}

// One 8-bit digit (bits shift .. shift + 7) of both selections of every set: histogram of the digit over the keys whose
// higher digits equal the prefix found so far.  Integer atomics only (shared, then one global add per non-empty bin).
constexpr int kSelThreads = 256;
__global__ void __launch_bounds__(kSelThreads) radix_hist_kernel(const unsigned long long* __restrict__ keys,
                                                                 long long set_stride, const unsigned long long* __restrict__ cnt,
                                                                 const unsigned long long* __restrict__ sel, int shift,
                                                                 unsigned* __restrict__ hist) {
    __shared__ unsigned sh[2 * 256];
    const int set = blockIdx.y;
    for (int j = threadIdx.x; j < 512; j += kSelThreads) sh[j] = 0;
    __syncthreads();
    const long long n = (long long)cnt[3 * set];
    const unsigned long long p0 = sel[4 * set], p1 = sel[4 * set + 2];
    const unsigned long long hmask = shift >= 56 ? 0ull : (~0ull << (shift + 8));
    const unsigned long long* k = keys + (long long)set * set_stride;
    for (long long i = (long long)blockIdx.x * kSelThreads + threadIdx.x; i < n; i += (long long)gridDim.x * kSelThreads) {
        const unsigned long long key = k[i];
        const unsigned dig = (unsigned)(key >> shift) & 255u;
        if (((key ^ p0) & hmask) == 0) atomicAdd(sh + dig, 1u);
        if (((key ^ p1) & hmask) == 0) atomicAdd(sh + 256 + dig, 1u);
    }
    __syncthreads();
    for (int j = threadIdx.x; j < 512; j += kSelThreads)
        if (sh[j]) atomicAdd(hist + 512LL * set + j, sh[j]);
}

// One CTA per selection: the bin that holds the rank extends the prefix; the histogram is cleared for the next digit.
__global__ void __launch_bounds__(256) radix_pick_kernel(unsigned* __restrict__ hist, unsigned long long* __restrict__ sel,
                                                         int shift) {
    __shared__ unsigned long long wsum[8];
    const int item = blockIdx.x, t = threadIdx.x, lane = t & 31, wid = t >> 5;
    unsigned* hb = hist + 256LL * item;
    const unsigned long long c = hb[t];
    hb[t] = 0;
    const unsigned long long rank = sel[2 * item + 1];
    unsigned long long x = c;                      // inclusive scan of the 256 bins
    for (int off = 1; off < 32; off <<= 1) {
        const unsigned long long y = __shfl_up_sync(0xffffffffu, x, off);
        if (lane >= off) x += y;
    }
    if (lane == 31) wsum[wid] = x;
    __syncthreads();
    for (int k = 0; k < wid; ++k) x += wsum[k];
    const unsigned long long excl = x - c;
    if (c && excl <= rank && rank < x) {
        sel[2 * item] |= (unsigned long long)t << shift;
        sel[2 * item + 1] = rank - excl;
    }
}

// One CTA per volume p: out[k][p] for k = dice, hausdorff, hausdorff_percentile, assd, surface_dice.  Set 2p holds the
// distances from the target's edges to the prediction's surface (d(T->P)), set 2p + 1 those of d(P->T).
__global__ void __launch_bounds__(256) surface_finalize_kernel(const unsigned long long* __restrict__ stats,
                                                               const unsigned long long* __restrict__ cnt,
                                                               const unsigned long long* __restrict__ sel,
                                                               const double* __restrict__ partial, int parts, int pairs,
                                                               double percentile, int weighted, double* __restrict__ out) {
    __shared__ double ssum[8];
    const int p = blockIdx.x;
    double sum = 0.0;                              // fixed order: strided per thread, warp tree, warps in order
    for (int i = threadIdx.x; i < 2 * parts; i += 256) sum += partial[2LL * p * parts + i];
    sum = warp_sum(sum);
    if ((threadIdx.x & 31) == 0) ssum[threadIdx.x >> 5] = sum;
    __syncthreads();
    if (threadIdx.x) return;
    for (int k = 1; k < 8; ++k) sum += ssum[k];
    const unsigned long long* st = stats + 5LL * p;
    const unsigned long long np = st[0], nt = st[1], ni = st[2], ep = st[3], et = st[4];
    const double nan = __longlong_as_double(0x7ff8000000000000LL), inf = __longlong_as_double(0x7ff0000000000000LL);
    double dice, hd, hp, assd, sdice;
    if (np == 0 && nt == 0) {
        dice = hd = hp = assd = sdice = nan;
    } else if (np == 0 || nt == 0) {
        dice = sdice = 0.0;
        hd = hp = assd = inf;
    } else {
        dice = __ddiv_rn((double)(2 * ni), (double)(np + nt));
        const unsigned long long* c0 = cnt + 6LL * p;      // set 2p
        const unsigned long long* c1 = c0 + 3;              // set 2p + 1
        hd = key_distance(max(c0[1], c1[1]), weighted);
        double pct[2];
        for (int s = 0; s < 2; ++s) {
            const long long set = 2LL * p + s;
            unsigned long long lo, hi;
            double g;
            pct_index(cnt[3 * set], percentile, lo, hi, g);
            pct[s] = np_lerp(key_distance(sel[4 * set], weighted), key_distance(sel[4 * set + 2], weighted), g);
        }
        hp = max(pct[0], pct[1]);
        assd = __ddiv_rn(sum, (double)(c0[0] + c1[0]));
        sdice = __ddiv_rn((double)(c0[2] + c1[2]), (double)(ep + et));
    }
    out[p] = dice;
    out[pairs + p] = hd;
    out[2 * pairs + p] = hp;
    out[3 * pairs + p] = assd;
    out[4 * pairs + p] = sdice;
}

template <int C>
static int launch_masks(const float* pred, const float* target, int b, long long spatial, unsigned char* pm, unsigned char* tm,
                        double* counts, cudaStream_t st) {
    const int blocks = (int)min((long long)2048, (spatial + kMetThreads - 1) / kMetThreads);
    seg_masks_kernel<C><<<dim3(blocks, b), kMetThreads, 0, st>>>(pred, target, spatial, pm, tm, counts);
    return check_launch("seg_masks_kernel");
}

}  // namespace ctu

using namespace ctu;

extern "C" int ctu_dice_coeff(const float* pred, const float* target, int b, int c, long long spatial, double* counts,
                              float* out, ctu_stream stream) {
    CTU_REQUIRE(pred && target && counts && out, "ctu_dice_coeff: null pointer");
    CTU_REQUIRE(b >= 1 && spatial >= 1 && c >= 2 && c <= 4, "ctu_dice_coeff: b=%d c=%d (2..4 channels)", b, c);
    cudaStream_t st = (cudaStream_t)stream;
    cudaMemsetAsync(counts, 0, sizeof(double) * 3 * b * (c - 1), st);
    int rc = c == 2 ? launch_masks<2>(pred, target, b, spatial, nullptr, nullptr, counts, st)
           : c == 3 ? launch_masks<3>(pred, target, b, spatial, nullptr, nullptr, counts, st)
                    : launch_masks<4>(pred, target, b, spatial, nullptr, nullptr, counts, st);
    if (rc) return rc;
    dice_coeff_finalize_kernel<<<1, 1, 0, st>>>(counts, b * (c - 1), out);
    return check_launch("dice_coeff_finalize_kernel");
}

extern "C" long long ctu_hausdorff_workspace_bytes(int b, int c, int d, int h, int w) {
    if (b < 1 || c < 2 || d < 1 || h < 1 || w < 1) return -1;
    const long long sets = 2LL * b * (c - 1), spatial = (long long)d * h * w;
    // masks + edges (1 B each) + two int32 distance planes per set, + counts / stats / maxima
    return sets * spatial * (2 + 8) + 16384 + 64LL * sets;
}

// Both min-plus passes of one EDT; the last one reduces in MODE.  Dynamic shared memory up to a 1024-long column tile.
template <typename T, int MODE>
static void axis_smem_attr() {
    static bool done = false;
    if (!done) {
        cudaFuncSetAttribute(edt_axis_kernel<T, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             1024 * Dist<T>::kLanes * (int)sizeof(T));
        done = true;
    }
}

// edges [sets][d][h][w] -> g0 (pass 1 along w) -> g1 (pass 2 along h) -> pass 3 along d, reduced in MODE.
// w3 / w2 / w1 = the axis weights of d / h / w (unused by the int path).
template <typename T, int MODE>
static int run_edt(const unsigned char* edges, T* g0, T* g1, int sets, int d, int h, int w, T w3, T w2, T w1, int* maxd2,
                   SurfAcc acc, cudaStream_t st) {
    constexpr int LN = Dist<T>::kLanes, TY = 256 / LN;
    const long long spatial = (long long)d * h * w;
    {   // pass 1 along w (all sets at once: rows = sets * d * h)
        const long long rows = (long long)sets * d * h;
        const int tx = w >= 128 ? 128 : (w >= 64 ? 64 : 32), ty = 256 / tx;
        edt_row_kernel<T><<<(unsigned)((rows + ty - 1) / ty), dim3(tx, ty), (size_t)ty * w, st>>>(edges, g0, w, rows, w1);
        if (int rc = check_launch("edt_row_kernel")) return rc;
    }
    axis_smem_attr<T, kStore>();
    axis_smem_attr<T, MODE>();
    // pass 2 along h: [outer = d][L = h][inner = w]
    const long long tiles = (w + LN - 1) / LN;
    edt_axis_kernel<T, kStore><<<dim3((unsigned)(d * tiles), 1, sets), dim3(LN, TY), (size_t)h * LN * sizeof(T), st>>>(
        g0, g1, h, w, d, spatial, w2, nullptr, nullptr, SurfAcc{});
    if (int rc = check_launch("edt_axis_kernel<h>")) return rc;
    // pass 3 along d: [outer = 1][L = d][inner = h*w], fused with the reduction over the partner's edge voxels
    const long long tiles3 = ((long long)h * w + LN - 1) / LN;
    edt_axis_kernel<T, MODE><<<dim3((unsigned)tiles3, 1, sets), dim3(LN, TY), (size_t)d * LN * sizeof(T), st>>>(
        g1, nullptr, d, (long long)h * w, 1, spatial, w3, edges, maxd2, acc);
    return check_launch("edt_axis_kernel<d>");
}

extern "C" int ctu_hausdorff(const float* pred, const float* target, int b, int c, int d, int h, int w, double inf_alt,
                             void* workspace, long long workspace_bytes, double* out, ctu_stream stream) {
    CTU_REQUIRE(pred && target && workspace && out, "ctu_hausdorff: null pointer");
    CTU_REQUIRE(b >= 1 && c >= 2 && c <= 4, "ctu_hausdorff: b=%d c=%d (2..4 channels)", b, c);
    CTU_REQUIRE(d >= 1 && h >= 1 && w >= 1 && d <= 1024 && h <= 1024 && w <= 1024, "ctu_hausdorff: dims %dx%dx%d (<= 1024)", d, h, w);
    CTU_REQUIRE(workspace_bytes >= ctu_hausdorff_workspace_bytes(b, c, d, h, w), "ctu_hausdorff: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    const long long spatial = (long long)d * h * w;
    const int pairs = b * (c - 1), sets = 2 * pairs;
    // workspace carving.  Set order: interleave (prediction, target) per pair so that partner(set) = set ^ 1.
    char* p = (char*)workspace;
    double* counts = (double*)p;              p += 2048;
    int* maxd2 = (int*)p;                     p += 1024;
    unsigned long long* stats = (unsigned long long*)p; p += 5 * 8 * 128;
    p += 64LL * sets;                         // slack (keeps the planes 64-byte aligned for any set count)
    p = (char*)(((uintptr_t)p + 255) & ~(uintptr_t)255);
    unsigned char* masks = (unsigned char*)p; p += sets * spatial;
    unsigned char* edges = (unsigned char*)p; p += sets * spatial;
    p = (char*)(((uintptr_t)p + 255) & ~(uintptr_t)255);
    int* g0 = (int*)p;                        p += sets * spatial * 4;
    int* g1 = (int*)p;
    CTU_REQUIRE(3 * pairs * sizeof(double) <= 2048 && sets * sizeof(int) <= 1024, "ctu_hausdorff: too many (batch, class) pairs");
    cudaMemsetAsync(workspace, 0, 2048 + 1024 + 5 * 8 * 128, st);
    // masks: kernel writes [b][c-1][spatial] for predictions and targets separately; interleave by using strided bases:
    // prediction mask of pair i at set 2i, target mask at set 2i+1  ->  write through two temporaries = the g1 plane
    unsigned char* pm = (unsigned char*)g1;
    unsigned char* tm = pm + (long long)pairs * spatial;
    int rc = c == 2 ? launch_masks<2>(pred, target, b, spatial, pm, tm, counts, st)
           : c == 3 ? launch_masks<3>(pred, target, b, spatial, pm, tm, counts, st)
                    : launch_masks<4>(pred, target, b, spatial, pm, tm, counts, st);
    if (rc) return rc;
    cudaMemcpy2DAsync(masks, 2 * spatial, pm, spatial, spatial, pairs, cudaMemcpyDeviceToDevice, st);
    cudaMemcpy2DAsync(masks + spatial, 2 * spatial, tm, spatial, spatial, pairs, cudaMemcpyDeviceToDevice, st);
    const int blocks = (int)min((long long)1024, (spatial + kMetThreads - 1) / kMetThreads);
    mask_edges_kernel<unsigned char, unsigned char><<<dim3(blocks, pairs), kMetThreads, 0, st>>>(
        masks, 2 * spatial, masks + spatial, 2 * spatial, edges, d, h, w, stats);
    if ((rc = check_launch("mask_edges_kernel"))) return rc;
    if ((rc = run_edt<int, kMax>(edges, g0, g1, sets, d, h, w, 1, 1, 1, maxd2, SurfAcc{}, st))) return rc;
    hausdorff_finalize_kernel<<<1, 1, 0, st>>>(maxd2, stats, pairs, inf_alt, out);
    return check_launch("hausdorff_finalize_kernel");
}

// ---------------------------------------------------------------- surface metrics
// Workspace: a zeroed head {stats [b][5], cnt [2b][3], sel [2b][2][2] (u64), hist [2b][2][256] (u32)}, the per-CTA
// distance sums [2b][parts], edges [2b][V] (1 B), g0 [2b][V] (8 B: the int or double plane of pass 1, then the key list
// of pass 3), g1 [2b][V] (the plane of pass 2: 4 B int, 8 B double).
struct SurfWs {
    unsigned long long *stats, *cnt, *sel;
    unsigned* hist;
    double* partial;
    unsigned char* edges;
    void *g0, *g1;
    long long head_bytes;
    int parts;
};

static bool surf_dims_ok(int b, int d, int h, int w) {
    return b >= 1 && d >= 1 && h >= 1 && w >= 1 && d <= 1024 && h <= 1024 && w <= 1024 && (long long)b * d * h * w < (1LL << 31);
}

static long long surf_layout(int b, int d, int h, int w, bool weighted, char* base, SurfWs* ws) {
    const long long sets = 2LL * b, spatial = (long long)d * h * w;
    const int lanes = weighted ? Dist<double>::kLanes : Dist<int>::kLanes;
    const int parts = cdiv((long long)h * w, lanes);
    const long long head = 8 * (5LL * b + 3 * sets + 4 * sets) + 4 * 512 * sets;
    long long off = 0;
    auto take = [&](long long bytes) { char* q = base + off; off += (bytes + 255) / 256 * 256; return q; };
    char* h0 = take(head);
    char* p1 = take(8LL * sets * parts);
    char* p2 = take(sets * spatial);
    char* p3 = take(8 * sets * spatial);
    char* p4 = take((weighted ? 8 : 4) * sets * spatial);
    if (ws) {
        ws->stats = (unsigned long long*)h0;
        ws->cnt = ws->stats + 5LL * b;
        ws->sel = ws->cnt + 3 * sets;
        ws->hist = (unsigned*)(ws->sel + 4 * sets);
        ws->partial = (double*)p1;
        ws->edges = (unsigned char*)p2;
        ws->g0 = p3;
        ws->g1 = p4;
        ws->head_bytes = head;
        ws->parts = parts;
    }
    return off;
}

template <typename TP, typename TT>
static int launch_surface_edges(const void* pred, const void* target, int b, int d, int h, int w, const SurfWs& ws,
                                cudaStream_t st) {
    const long long spatial = (long long)d * h * w;
    const int blocks = (int)min((long long)1024, (spatial + kMetThreads - 1) / kMetThreads);
    mask_edges_kernel<TP, TT><<<dim3(blocks, b), kMetThreads, 0, st>>>((const TP*)pred, spatial, (const TT*)target, spatial,
                                                                       ws.edges, d, h, w, ws.stats);
    return check_launch("mask_edges_kernel");
}

extern "C" long long ctu_surface_metrics_workspace_bytes(int b, int d, int h, int w, int weighted) {
    if (!surf_dims_ok(b, d, h, w)) return -1;
    return surf_layout(b, d, h, w, weighted != 0, nullptr, nullptr);
}

extern "C" int ctu_surface_metrics(int pred_dtype, const void* pred, int target_dtype, const void* target, int b, int d, int h,
                                   int w, const double* spacing, double percentile, double tolerance, double* out, void* ws_ptr,
                                   long long ws_bytes, ctu_stream stream) {
    CTU_REQUIRE(pred && target && out && ws_ptr, "ctu_surface_metrics: null pointer");
    CTU_REQUIRE((pred_dtype == CTU_MASK_U8 || pred_dtype == CTU_MASK_F32) &&
                    (target_dtype == CTU_MASK_U8 || target_dtype == CTU_MASK_F32),
                "ctu_surface_metrics: dtypes %d / %d (CTU_MASK_U8 or CTU_MASK_F32)", pred_dtype, target_dtype);
    CTU_REQUIRE(surf_dims_ok(b, d, h, w), "ctu_surface_metrics: shape %dx%dx%dx%d (each axis 1..1024, fewer than 2^31 voxels)",
                b, d, h, w);
    if (spacing)
        for (int i = 0; i < 3; ++i)
            CTU_REQUIRE(spacing[i] > 0 && spacing[i] < HUGE_VAL, "ctu_surface_metrics: spacing[%d] = %g (positive, finite)", i,
                        spacing[i]);
    CTU_REQUIRE(percentile >= 0 && percentile <= 100, "ctu_surface_metrics: percentile %g (0..100)", percentile);
    CTU_REQUIRE(tolerance >= 0, "ctu_surface_metrics: tolerance %g (>= 0)", tolerance);
    const bool weighted = spacing != nullptr;
    CTU_REQUIRE(((uintptr_t)ws_ptr & 7) == 0, "ctu_surface_metrics: workspace must be 8-byte aligned");
    CTU_REQUIRE(ws_bytes >= ctu_surface_metrics_workspace_bytes(b, d, h, w, weighted),
                "ctu_surface_metrics: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    SurfWs ws;
    surf_layout(b, d, h, w, weighted, (char*)ws_ptr, &ws);
    const int sets = 2 * b;
    const long long spatial = (long long)d * h * w;
    cudaError_t e = cudaMemsetAsync(ws_ptr, 0, ws.head_bytes, st);
    if (e != cudaSuccess) {
        set_error("ctu_surface_metrics: memset: %s", cudaGetErrorString(e));
        return (int)e;
    }
    const bool pu8 = pred_dtype == CTU_MASK_U8, tu8 = target_dtype == CTU_MASK_U8;
    int rc = pu8 ? (tu8 ? launch_surface_edges<unsigned char, unsigned char>(pred, target, b, d, h, w, ws, st)
                        : launch_surface_edges<unsigned char, float>(pred, target, b, d, h, w, ws, st))
                 : (tu8 ? launch_surface_edges<float, unsigned char>(pred, target, b, d, h, w, ws, st)
                        : launch_surface_edges<float, float>(pred, target, b, d, h, w, ws, st));
    if (rc) return rc;
    const SurfAcc acc{(unsigned long long*)ws.g0, ws.cnt, ws.partial, tolerance};
    if (weighted) {
        const double s2[3] = {spacing[0] * spacing[0], spacing[1] * spacing[1], spacing[2] * spacing[2]};
        rc = run_edt<double, kSurface>(ws.edges, (double*)ws.g0, (double*)ws.g1, sets, d, h, w, s2[0], s2[1], s2[2], nullptr,
                                       acc, st);
    } else {
        rc = run_edt<int, kSurface>(ws.edges, (int*)ws.g0, (int*)ws.g1, sets, d, h, w, 1, 1, 1, nullptr, acc, st);
    }
    if (rc) return rc;
    pct_rank_kernel<<<cdiv(2 * sets, 256), 256, 0, st>>>(ws.cnt, sets, percentile, ws.sel);
    if ((rc = check_launch("pct_rank_kernel"))) return rc;
    // int keys are below 2^31: 4 digits; double keys: 8
    const unsigned hblocks = (unsigned)min((long long)1024, (spatial + kSelThreads - 1) / kSelThreads);
    for (int shift = weighted ? 56 : 24; shift >= 0; shift -= 8) {
        radix_hist_kernel<<<dim3(hblocks, sets), kSelThreads, 0, st>>>((const unsigned long long*)ws.g0, spatial, ws.cnt, ws.sel, shift, ws.hist);
        radix_pick_kernel<<<2 * sets, 256, 0, st>>>(ws.hist, ws.sel, shift);
    }
    if ((rc = check_launch("radix_hist/pick_kernel"))) return rc;
    surface_finalize_kernel<<<b, 256, 0, st>>>(ws.stats, ws.cnt, ws.sel, ws.partial, ws.parts, b, percentile, weighted, out);
    return check_launch("surface_finalize_kernel");
}
