// Connected-component labelling of binary volumes (scipy.ndimage.label semantics) and the largest-component /
// small-component filters built on it.  The reference has no post-processing of its label volumes; the semantics are
// frozen by tests/components_oracle.py (scipy.ndimage.label + numpy.bincount) and every output is compared bit for bit.
//
// A voxel is foreground when it is non-zero.  parent[] holds int32 GLOBAL linear indices i = b*V + (z*H + y)*W + x over
// the whole batch (B*V < 2^31); no union ever joins voxels of two volumes, so every tree stays inside its volume.
//
//   1. ccl_local_kernel     one CTA per 8 x 8 x 32 (z, y, x) tile: union-find on tile-local indices in shared memory,
//                           then parent[i] = global index of the tile-local root (background: kBg).  The filter path
//                           also zeroes size[] at every tile-local root (the global roots are among them).
//   2. ccl_boundary_kernel  one CTA per tile: every foreground voxel on a lower face of its tile (local z, y or x = 0)
//                           unions with its neighbours across that face (global atomicMin union).  Every edge between two
//                           tiles has one end on a lower face of its own tile, so every such edge is seen.
//   3. ccl_flatten_kernel   one CTA per chunk of 4096 consecutive voxels of one volume (raster order): parent[i] = root;
//                           a root gets -1 - (its rank among the chunk's roots); chunk_roots[c] = the chunk's root count.
//                           The filter path adds the component sizes here.
//   4. ccl_scan_kernel      one CTA per volume: exclusive scan of chunk_roots (the segmented scan) and counts[b].
//   5. ccl_labels_kernel    labels[i] = 1 + chunk_off[chunk(root)] + rank of the root in its chunk.
//   The filters skip 4 and 5: ccl_select_kernel (largest component only) reduces max(size << 32 | ~root) per volume,
//   ccl_filter_kernel writes the output in one pass.
//
// Invariants
//   * The root is the smallest index.  A parent index is never larger than its child: both unions link the larger root
//     under the smaller with atomicMin, and flattening only replaces a parent by an ancestor.  Every find therefore walks
//     strictly decreasing indices and terminates, and every component's root is its smallest linear index, i.e. its
//     first voxel in raster order: numbering the roots in raster order gives scipy's numbering.
//   * No spin-waits across CTAs and no grid-wide barrier: passes are separated by kernel boundaries only.  A union
//     retries only after its atomicMin found the root already linked, and then continues from the (strictly smaller)
//     value it found, so every loop is bounded by the index range whatever the input.
//   * Contended atomics: the skull is one component of 10^6..10^7 voxels.  Sizes are summed per thread (runs of equal
//     roots), then per CTA in a 64-slot shared-memory table, and only then added to size[root]: one global atomic per
//     (CTA, root) instead of one per voxel.
//   * Vectorised I/O: with W % 16 == 0 (tiles) or V % 16 == 0 (chunks) and 16-byte aligned buffers, mask reads, parent
//     and label reads / writes and the filter output use 16-byte accesses; otherwise the same kernels go voxel by voxel.
#include "common.cuh"

namespace ctu {

constexpr int kCclThreads = 256;
constexpr int kTZ = 8, kTY = 8, kTX = 32, kTile = kTZ * kTY * kTX;     // 2048 voxels, 8 per thread
constexpr int kChunk = 4096;                                             // 16 voxels per thread
constexpr int kBg = 0x7fffffff;                                          // parent[] of a background voxel
constexpr int kFaceVox = kTY * kTX + (kTZ - 1) * kTX + (kTZ - 1) * (kTY - 1);   // z = 0 plane, y = 0 rows, x = 0 column

// The backward half of the 26-neighbourhood (raster offset < 0), (dz, dy, dx): the first 3 are the 6-neighbourhood, the
// first 9 the 18-neighbourhood (scipy.ndimage.generate_binary_structure(3, r), r = 1, 2, 3).
__device__ __forceinline__ void nbr(int k, int& dz, int& dy, int& dx) {
    constexpr int oz[13] = {0, 0, -1, 0, 0, -1, -1, -1, -1, -1, -1, -1, -1};
    constexpr int oy[13] = {0, -1, 0, -1, -1, -1, 1, 0, 0, -1, -1, 1, 1};
    constexpr int ox[13] = {-1, 0, 0, -1, 1, 0, 0, -1, 1, -1, 1, -1, 1};
    dz = oz[k], dy = oy[k], dx = ox[k];
}
template <int CONN> struct NbrCount { static constexpr int n = CONN == 6 ? 3 : (CONN == 18 ? 9 : 13); };

// ---------------------------------------------------------------- union-find (Playne & Hawick 2018)
// find: parents only decrease along a path, so the walk terminates.  Negative entries are the root marks written by
// ccl_flatten_kernel (only ever read while that kernel runs).
__device__ __forceinline__ int sfind(volatile int* L, int x) {
    int p;
    while ((p = L[x]) != x) x = p;
    return x;
}
__device__ __forceinline__ void sunion(int* L, int a, int b) {
    while (true) {
        a = sfind(L, a);
        b = sfind(L, b);
        if (a == b) return;
        if (a > b) { const int t = a; a = b; b = t; }
        const int old = atomicMin(L + b, a);   // link the larger root under the smaller
        if (old == b) return;
        b = old;                               // b was linked meanwhile: join a with what it was linked to
    }
}
__device__ __forceinline__ int gfind(const int* parent, int x) {
    while (true) {
        const int p = __ldcg(parent + x);      // L2: the entries change under concurrent unions / flattening
        if (p < 0 || p == x) return x;
        x = p;
    }
}
__device__ __forceinline__ void gunion(int* parent, int a, int b) {
    while (true) {
        a = gfind(parent, a);
        b = gfind(parent, b);
        if (a == b) return;
        if (a > b) { const int t = a; a = b; b = t; }
        const int old = atomicMin(parent + b, a);
        if (old == b) return;
        b = old;
    }
}

__device__ __forceinline__ bool nonzero(unsigned char v) { return v != 0; }
__device__ __forceinline__ bool nonzero(float v) { return v != 0.0f; }    // NaN counts as foreground, -0.0 does not

struct TileGeo {
    int b, z0, y0, x0, vbase;
};
__device__ __forceinline__ TileGeo tile_geo(int ty_n, int tx_n, int tiles_per_vol, int V) {
    TileGeo g;
    g.b = blockIdx.x / tiles_per_vol;
    int r = blockIdx.x - g.b * tiles_per_vol;
    const int tz = r / (ty_n * tx_n);
    r -= tz * ty_n * tx_n;
    const int ty = r / tx_n;
    g.z0 = tz * kTZ, g.y0 = ty * kTY, g.x0 = (r - ty * tx_n) * kTX;
    g.vbase = g.b * V;
    return g;
}

// ---------------------------------------------------------------- 1. local merge
// Thread t owns the 8 consecutive x voxels lt = 8t .. 8t + 7 of the tile (lt = (lz * 8 + ly) * 32 + lx): the tile-local
// raster order agrees with the global one, so the smallest local index of a local component is its smallest global index.
template <int CONN, typename T, bool VEC>
__global__ void __launch_bounds__(kCclThreads) ccl_local_kernel(const T* __restrict__ in, int d, int h, int w, int ty_n,
                                                                int tx_n, int tiles_per_vol, int* __restrict__ parent,
                                                                int* __restrict__ size) {
    __shared__ int L[kTile];
    const TileGeo g = tile_geo(ty_n, tx_n, tiles_per_vol, d * h * w);
    const T* vin = in + g.vbase;
    if (VEC) {   // w % 16 == 0: a 16-voxel row segment is entirely inside or entirely outside the volume
        constexpr int per = 16 / sizeof(T);                          // voxels per 16-byte load
        constexpr int nseg = kTile / per;
        for (int s = threadIdx.x; s < nseg; s += kCclThreads) {
            const int lt = s * per, lz = lt >> 8, ly = (lt >> 5) & 7, lx = lt & 31;
            const int z = g.z0 + lz, y = g.y0 + ly, x = g.x0 + lx;
            uint4 u = make_uint4(0, 0, 0, 0);
            if (z < d && y < h && x < w) u = __ldg(reinterpret_cast<const uint4*>(vin + ((long long)z * h + y) * w + x));
            const uint32_t word[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
            for (int j = 0; j < per; ++j) {
                bool fg;
                if constexpr (sizeof(T) == 1) fg = ((word[j >> 2] >> (8 * (j & 3))) & 0xffu) != 0;
                else fg = nonzero(__uint_as_float(word[j]));
                L[lt + j] = fg ? lt + j : -1;
            }
        }
    } else {
        for (int lt = threadIdx.x; lt < kTile; lt += kCclThreads) {
            const int z = g.z0 + (lt >> 8), y = g.y0 + ((lt >> 5) & 7), x = g.x0 + (lt & 31);
            const bool fg = z < d && y < h && x < w && nonzero(vin[((long long)z * h + y) * w + x]);
            L[lt] = fg ? lt : -1;
        }
    }
    __syncthreads();
    const int t0 = threadIdx.x * 8, lz = t0 >> 8, ly = (t0 >> 5) & 7, lx0 = t0 & 31;
#pragma unroll 1
    for (int j = 0; j < 8; ++j) {
        const int lt = t0 + j, lx = lx0 + j;
        if (L[lt] < 0) continue;                                     // background stays -1; unions write only >= 0
#pragma unroll
        for (int k = 0; k < NbrCount<CONN>::n; ++k) {
            int dz, dy, dx;
            nbr(k, dz, dy, dx);
            if (lz + dz < 0 || ly + dy < 0 || ly + dy >= kTY || lx + dx < 0 || lx + dx >= kTX) continue;
            const int ln = lt + (dz * kTY + dy) * kTX + dx;
            if (L[ln] >= 0) sunion(L, lt, ln);
        }
    }
    __syncthreads();
    const int z = g.z0 + lz, y = g.y0 + ly, x0 = g.x0 + lx0;
    if (z >= d || y >= h) return;
    const int row = g.vbase + (z * h + y) * w;
    int v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        v[j] = kBg;
        if (L[t0 + j] >= 0) {
            const int rt = sfind(L, t0 + j);
            v[j] = g.vbase + ((g.z0 + (rt >> 8)) * h + g.y0 + ((rt >> 5) & 7)) * w + g.x0 + (rt & 31);
            if (size && rt == t0 + j) size[v[j]] = 0;
        }
    }
    if (VEC) {
        if (x0 < w) {                                                // w % 16 == 0: all 8 inside
            int4* p = reinterpret_cast<int4*>(parent + row + x0);
            p[0] = make_int4(v[0], v[1], v[2], v[3]);
            p[1] = make_int4(v[4], v[5], v[6], v[7]);
        }
    } else {
#pragma unroll
        for (int j = 0; j < 8; ++j)
            if (x0 + j < w) parent[row + x0 + j] = v[j];
    }
}

// ---------------------------------------------------------------- 2. boundary merge
// An edge between two tiles differs by one along an axis where one end sits at local coordinate 0 of its tile; that end
// checks its neighbours one step back along such an axis.  Duplicate checks (a voxel on two lower faces) are harmless.
template <int CONN>
__global__ void __launch_bounds__(kCclThreads) ccl_boundary_kernel(int d, int h, int w, int ty_n, int tx_n, int tiles_per_vol,
                                                                   int* __restrict__ parent) {
    const TileGeo g = tile_geo(ty_n, tx_n, tiles_per_vol, d * h * w);
    for (int k = threadIdx.x; k < kFaceVox; k += kCclThreads) {
        int lz, ly, lx;
        if (k < kTY * kTX) lz = 0, ly = k >> 5, lx = k & 31;
        else if (k < kTY * kTX + (kTZ - 1) * kTX) lz = 1 + ((k - kTY * kTX) >> 5), ly = 0, lx = (k - kTY * kTX) & 31;
        else {
            const int r = k - kTY * kTX - (kTZ - 1) * kTX;
            lz = 1 + r / (kTY - 1), ly = 1 + r % (kTY - 1), lx = 0;
        }
        const int z = g.z0 + lz, y = g.y0 + ly, x = g.x0 + lx;
        if (z >= d || y >= h || x >= w) continue;
        const int i = g.vbase + (z * h + y) * w + x;
        if (__ldcg(parent + i) == kBg) continue;
#pragma unroll
        for (int n = 0; n < 2 * NbrCount<CONN>::n; ++n) {
            int dz, dy, dx;
            nbr(n >> 1, dz, dy, dx);
            if (n & 1) dz = -dz, dy = -dy, dx = -dx;                // the forward half
            const bool crosses = (lz == 0 && dz < 0) || (ly == 0 && dy < 0) || (lx == 0 && dx < 0);
            if (!crosses || z + dz < 0 || z + dz >= d || y + dy < 0 || y + dy >= h || x + dx < 0 || x + dx >= w) continue;
            const int j = i + (dz * h + dy) * w + dx;
            if (__ldcg(parent + j) != kBg) gunion(parent, i, j);
        }
    }
}

// ---------------------------------------------------------------- chunk helpers
// Thread t of the chunk's CTA owns voxels i0 .. i0 + 15, of which n (possibly <= 0) lie inside the volume; i0 is only
// formed when n > 0, so no index past the last voxel of the batch is computed.
struct ChunkGeo {
    int b, c, i0, n;
};
__device__ __forceinline__ ChunkGeo chunk_geo(int V, int cpv) {
    ChunkGeo g;
    g.c = blockIdx.x;
    g.b = g.c / cpv;
    const int k = g.c - g.b * cpv, first = k * kChunk + threadIdx.x * 16;
    g.n = min(V - k * kChunk, kChunk) - threadIdx.x * 16;
    g.i0 = g.n > 0 ? g.b * V + first : 0;
    return g;
}
// 16 int32 of voxels [i0, i0 + 16), n of them valid (VEC: a chunk is a whole number of 16-voxel groups)
template <bool VEC>
__device__ __forceinline__ void load16(const int* __restrict__ p, int i0, int n, int (&v)[16]) {
    if (VEC) {
        if (n > 0) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int4 a = reinterpret_cast<const int4*>(p + i0)[q];
                v[4 * q] = a.x, v[4 * q + 1] = a.y, v[4 * q + 2] = a.z, v[4 * q + 3] = a.w;
            }
        } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = kBg;
        }
    } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = j < n ? p[i0 + j] : kBg;
    }
}
template <bool VEC>
__device__ __forceinline__ void store16(int* __restrict__ p, int i0, int n, const int (&v)[16]) {
    if (VEC) {
        if (n > 0) {
#pragma unroll
            for (int q = 0; q < 4; ++q)
                reinterpret_cast<int4*>(p + i0)[q] = make_int4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
        }
    } else {
#pragma unroll
        for (int j = 0; j < 16; ++j)
            if (j < n) p[i0 + j] = v[j];
    }
}

__device__ __forceinline__ int block_exclusive_sum(int v, int& total) {
    __shared__ int warp_tot[kCclThreads / 32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) warp_tot[wid] = inc;
    __syncthreads();
    int off = 0;
    total = 0;
#pragma unroll
    for (int i = 0; i < kCclThreads / 32; ++i) {
        const int t = warp_tot[i];
        off += i < wid ? t : 0;
        total += t;
    }
    __syncthreads();
    return off + inc - v;
}

// ---------------------------------------------------------------- 3. flatten, rank roots per chunk, sizes
constexpr int kSizeSlots = 64;
__device__ __forceinline__ void size_add(int* keys, int* cnts, int* __restrict__ size, int r, int n) {
    int s = (int)(((unsigned)r * 0x9E3779B1u) >> 26);
#pragma unroll 1
    for (int probe = 0; probe < 8; ++probe) {
        const int k = atomicCAS(keys + s, -1, r);
        if (k == -1 || k == r) {
            atomicAdd(cnts + s, n);
            return;
        }
        s = (s + 1) & (kSizeSlots - 1);
    }
    atomicAdd(size + r, n);                                          // table crowded (many small components): direct
}

template <bool VEC, bool SIZES>
__global__ void __launch_bounds__(kCclThreads) ccl_flatten_kernel(int V, int cpv, int* __restrict__ parent,
                                                                  int* __restrict__ chunk_roots, int* __restrict__ size) {
    __shared__ int s_key[kSizeSlots], s_cnt[kSizeSlots];
    const ChunkGeo g = chunk_geo(V, cpv);
    if (SIZES && threadIdx.x < kSizeSlots) s_key[threadIdx.x] = -1, s_cnt[threadIdx.x] = 0;
    const int i0 = g.i0;
    int v[16];
    load16<VEC>(parent, i0, g.n, v);
    int nroots = 0;
    unsigned root_bits = 0;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        if (v[j] == kBg) continue;
        if (v[j] == i0 + j) root_bits |= 1u << j, ++nroots;
        else v[j] = gfind(parent, v[j]);
    }
    int total;
    int rank = block_exclusive_sum(nroots, total);                   // (its barrier also publishes the table reset)
#pragma unroll
    for (int j = 0; j < 16; ++j)
        if (root_bits >> j & 1) v[j] = -1 - rank++;
    store16<VEC>(parent, i0, g.n, v);
    if (threadIdx.x == 0) chunk_roots[g.c] = total;
    if (SIZES) {
        int cur = -1, n = 0;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            if (v[j] == kBg) continue;
            const int r = v[j] < 0 ? i0 + j : v[j];
            if (r != cur) {
                if (n) size_add(s_key, s_cnt, size, cur, n);
                cur = r, n = 0;
            }
            ++n;
        }
        if (n) size_add(s_key, s_cnt, size, cur, n);
        __syncthreads();
        if (threadIdx.x < kSizeSlots && s_key[threadIdx.x] >= 0) atomicAdd(size + s_key[threadIdx.x], s_cnt[threadIdx.x]);
    }
}

// ---------------------------------------------------------------- 4. per-volume exclusive scan of the root counts
__global__ void __launch_bounds__(kCclThreads) ccl_scan_kernel(const int* __restrict__ chunk_roots, int cpv,
                                                               int* __restrict__ chunk_off, long long* __restrict__ counts) {
    const int b = blockIdx.x;
    const int* in = chunk_roots + (long long)b * cpv;
    int* out = chunk_off + (long long)b * cpv;
    constexpr int kItems = 16;
    int carry = 0;
    for (int base = 0; base < cpv; base += kCclThreads * kItems) {
        const int k0 = base + threadIdx.x * kItems;
        int v[kItems], sum = 0;
#pragma unroll
        for (int j = 0; j < kItems; ++j) v[j] = k0 + j < cpv ? in[k0 + j] : 0, sum += v[j];
        int total;
        int off = carry + block_exclusive_sum(sum, total);
#pragma unroll
        for (int j = 0; j < kItems; ++j)
            if (k0 + j < cpv) out[k0 + j] = off, off += v[j];
        carry += total;
    }
    if (threadIdx.x == 0) counts[b] = carry;
}

// ---------------------------------------------------------------- 5. labels
template <bool VEC>
__global__ void __launch_bounds__(kCclThreads) ccl_labels_kernel(const int* __restrict__ parent, const int* __restrict__ chunk_off,
                                                                 int V, int cpv, int* __restrict__ labels) {
    const ChunkGeo g = chunk_geo(V, cpv);
    const int i0 = g.i0;
    int v[16];
    load16<VEC>(parent, i0, g.n, v);
    const int own = chunk_off[g.c];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const int p = v[j];
        if (p == kBg) v[j] = 0;
        else if (p < 0) v[j] = own - p;                               // 1 + own + (-1 - p)
        else v[j] = chunk_off[g.b * cpv + (p - g.b * V) / kChunk] - __ldg(parent + p);
    }
    store16<VEC>(labels, i0, g.n, v);
}

// ---------------------------------------------------------------- filters
__device__ __forceinline__ unsigned long long block_max_u64(unsigned long long v) {
    __shared__ unsigned long long warp_max[kCclThreads / 32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
    if ((threadIdx.x & 31) == 0) warp_max[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0)
        for (int i = 1; i < kCclThreads / 32; ++i) v = max(v, warp_max[i]);
    return v;
}

// best[b] = max over the volume's roots r of (size[r] << 32 | ~r): the largest component, ties to the smaller root
// (= the lower label).  0 = no foreground.
template <bool VEC>
__global__ void __launch_bounds__(kCclThreads) ccl_select_kernel(const int* __restrict__ parent, const int* __restrict__ size,
                                                                 int V, int cpv, unsigned long long* __restrict__ best) {
    const ChunkGeo g = chunk_geo(V, cpv);
    const int i0 = g.i0;
    int v[16];
    load16<VEC>(parent, i0, g.n, v);
    unsigned long long key = 0;
#pragma unroll
    for (int j = 0; j < 16; ++j)
        if (v[j] < 0) key = max(key, (unsigned long long)(unsigned)size[i0 + j] << 32 | (unsigned)~(i0 + j));
    key = block_max_u64(key);
    if (threadIdx.x == 0 && key) atomicMax(best + g.b, key);
}

// out = 0 on the voxels of dropped components, in everywhere else.  min_size < 0: keep the root chosen in best[b].
template <typename T, bool VEC>
__global__ void __launch_bounds__(kCclThreads) ccl_filter_kernel(const T* __restrict__ in, T* __restrict__ out,
                                                                 const int* __restrict__ parent, const int* __restrict__ size,
                                                                 const unsigned long long* __restrict__ best,
                                                                 long long min_size, int V, int cpv) {
    const ChunkGeo g = chunk_geo(V, cpv);
    const int i0 = g.i0;
    int v[16];
    load16<VEC>(parent, i0, g.n, v);
    int keep_root = -1;
    if (min_size < 0) {
        const unsigned long long k = best[g.b];
        keep_root = k ? (int)~(unsigned)(k & 0xffffffffu) : -1;
    }
    unsigned drop = 0;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        if (v[j] == kBg) continue;
        const int r = v[j] < 0 ? i0 + j : v[j];
        const bool keep = min_size < 0 ? r == keep_root : (long long)__ldg(size + r) >= min_size;
        if (!keep) drop |= 1u << j;
    }
    if (VEC) {
        if (g.n <= 0) return;
        constexpr int per = 16 / sizeof(T);
#pragma unroll
        for (int q = 0; q < 16 / per; ++q) {
            uint4 u = __ldg(reinterpret_cast<const uint4*>(in + i0) + q);
            uint32_t word[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
            for (int j = 0; j < per; ++j)
                if (drop >> (q * per + j) & 1) {
                    if constexpr (sizeof(T) == 1) word[j >> 2] &= ~(0xffu << (8 * (j & 3)));
                    else word[j] = 0;
                }
            reinterpret_cast<uint4*>(out + i0)[q] = make_uint4(word[0], word[1], word[2], word[3]);
        }
    } else {
#pragma unroll
        for (int j = 0; j < 16; ++j)
            if (j < g.n) out[i0 + j] = (drop >> j & 1) ? T(0) : in[i0 + j];
    }
}

// ---------------------------------------------------------------- host side
struct CclWs {
    int* parent;
    int* size;
    int* chunk_roots;
    int* chunk_off;
    unsigned long long* best;
};

static long long align256(long long x) { return (x + 255) & ~255LL; }

static bool ccl_dims_ok(int b, int d, int h, int w) {
    return b >= 1 && d >= 1 && h >= 1 && w >= 1 && (long long)b * d * h * w < (1LL << 31);
}

static long long ccl_layout(int b, int d, int h, int w, char* base, CclWs* ws) {
    const long long n = (long long)b * d * h * w, nchunks = (long long)b * cdiv((long long)d * h * w, kChunk);
    long long off = 0;
    auto take = [&](long long bytes) { char* p = base + off; off += align256(bytes); return p; };
    char* p0 = take(4 * n);
    char* p1 = take(4 * n);
    char* p2 = take(4 * nchunks);
    char* p3 = take(4 * nchunks);
    char* p4 = take(8LL * b);
    if (ws) *ws = {(int*)p0, (int*)p1, (int*)p2, (int*)p3, (unsigned long long*)p4};
    return off;
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

#define CTU_CCL_CONN(conn, ...)                       \
    do {                                              \
        if ((conn) == 6) {                            \
            constexpr int CONN = 6;                   \
            __VA_ARGS__;                              \
        } else if ((conn) == 18) {                    \
            constexpr int CONN = 18;                  \
            __VA_ARGS__;                              \
        } else {                                      \
            constexpr int CONN = 26;                  \
            __VA_ARGS__;                              \
        }                                             \
    } while (0)

// passes 1-3 (sizes: the filter path)
template <typename T>
static int ccl_core(const T* in, int b, int d, int h, int w, int conn, const CclWs& ws, bool sizes, bool vec_chunks,
                    cudaStream_t st) {
    const int V = d * h * w, cpv = cdiv(V, kChunk);
    const int tz_n = cdiv(d, kTZ), ty_n = cdiv(h, kTY), tx_n = cdiv(w, kTX), tpv = tz_n * ty_n * tx_n;
    const unsigned tiles = (unsigned)((long long)b * tpv), chunks = (unsigned)((long long)b * cpv);
    const bool vec_rows = w % 16 == 0 && aligned16(in) && aligned16(ws.parent);
    int* size = sizes ? ws.size : nullptr;
    CTU_CCL_CONN(conn, {
        if (vec_rows) ccl_local_kernel<CONN, T, true><<<tiles, kCclThreads, 0, st>>>(in, d, h, w, ty_n, tx_n, tpv, ws.parent, size);
        else ccl_local_kernel<CONN, T, false><<<tiles, kCclThreads, 0, st>>>(in, d, h, w, ty_n, tx_n, tpv, ws.parent, size);
        ccl_boundary_kernel<CONN><<<tiles, kCclThreads, 0, st>>>(d, h, w, ty_n, tx_n, tpv, ws.parent);
    });
    if (int rc = check_launch("ccl_local/boundary_kernel")) return rc;
    if (vec_chunks) {
        if (sizes) ccl_flatten_kernel<true, true><<<chunks, kCclThreads, 0, st>>>(V, cpv, ws.parent, ws.chunk_roots, ws.size);
        else ccl_flatten_kernel<true, false><<<chunks, kCclThreads, 0, st>>>(V, cpv, ws.parent, ws.chunk_roots, nullptr);
    } else {
        if (sizes) ccl_flatten_kernel<false, true><<<chunks, kCclThreads, 0, st>>>(V, cpv, ws.parent, ws.chunk_roots, ws.size);
        else ccl_flatten_kernel<false, false><<<chunks, kCclThreads, 0, st>>>(V, cpv, ws.parent, ws.chunk_roots, nullptr);
    }
    return check_launch("ccl_flatten_kernel");
}

}  // namespace ctu

using namespace ctu;

extern "C" long long ctu_components_workspace_bytes(int b, int d, int h, int w) {
    if (!ccl_dims_ok(b, d, h, w)) return -1;
    return ccl_layout(b, d, h, w, nullptr, nullptr);
}

#define CTU_CCL_CHECK(fn, in, out, in_dtype, b, d, h, w, conn, ws, ws_bytes)                                                \
    CTU_REQUIRE(in && out && ws, fn ": null pointer");                                                                      \
    CTU_REQUIRE(in_dtype == CTU_MASK_U8 || in_dtype == CTU_MASK_F32, fn ": in_dtype %d (CTU_MASK_U8 or CTU_MASK_F32)",      \
                in_dtype);                                                                                                  \
    CTU_REQUIRE(ccl_dims_ok(b, d, h, w), fn ": shape %dx%dx%dx%d (each >= 1, fewer than 2^31 voxels)", b, d, h, w);        \
    CTU_REQUIRE(conn == 6 || conn == 18 || conn == 26, fn ": connectivity %d (6, 18 or 26)", conn);                       \
    CTU_REQUIRE(ws_bytes >= ctu_components_workspace_bytes(b, d, h, w), fn ": workspace too small");                       \
    CTU_REQUIRE(aligned16(ws), fn ": workspace must be 16-byte aligned")

extern "C" int ctu_label_components(int in_dtype, const void* in, int b, int d, int h, int w, int connectivity, int* labels,
                                    long long* counts, void* ws_ptr, long long ws_bytes, ctu_stream stream) {
    CTU_CCL_CHECK("ctu_label_components", in, labels, in_dtype, b, d, h, w, connectivity, ws_ptr, ws_bytes);
    CTU_REQUIRE(counts, "ctu_label_components: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    CclWs ws;
    ccl_layout(b, d, h, w, (char*)ws_ptr, &ws);
    const int V = d * h * w, cpv = cdiv(V, kChunk);
    const unsigned chunks = (unsigned)((long long)b * cpv);
    const bool vec = V % 16 == 0 && aligned16(labels);
    int rc = in_dtype == CTU_MASK_U8
                 ? ccl_core((const unsigned char*)in, b, d, h, w, connectivity, ws, false, vec, st)
                 : ccl_core((const float*)in, b, d, h, w, connectivity, ws, false, vec, st);
    if (rc) return rc;
    ccl_scan_kernel<<<b, kCclThreads, 0, st>>>(ws.chunk_roots, cpv, ws.chunk_off, counts);
    if (vec) ccl_labels_kernel<true><<<chunks, kCclThreads, 0, st>>>(ws.parent, ws.chunk_off, V, cpv, labels);
    else ccl_labels_kernel<false><<<chunks, kCclThreads, 0, st>>>(ws.parent, ws.chunk_off, V, cpv, labels);
    return check_launch("ctu_label_components");
}

extern "C" int ctu_filter_components(int in_dtype, const void* in, int b, int d, int h, int w, int connectivity,
                                     long long min_size, void* out, void* ws_ptr, long long ws_bytes, ctu_stream stream) {
    CTU_CCL_CHECK("ctu_filter_components", in, out, in_dtype, b, d, h, w, connectivity, ws_ptr, ws_bytes);
    cudaStream_t st = (cudaStream_t)stream;
    CclWs ws;
    ccl_layout(b, d, h, w, (char*)ws_ptr, &ws);
    const int V = d * h * w, cpv = cdiv(V, kChunk);
    const unsigned chunks = (unsigned)((long long)b * cpv);
    const bool vec = V % 16 == 0 && aligned16(in) && aligned16(out);
    int rc = in_dtype == CTU_MASK_U8
                 ? ccl_core((const unsigned char*)in, b, d, h, w, connectivity, ws, true, vec, st)
                 : ccl_core((const float*)in, b, d, h, w, connectivity, ws, true, vec, st);
    if (rc) return rc;
    if (min_size < 0) {
        cudaError_t e = cudaMemsetAsync(ws.best, 0, 8LL * b, st);
        if (e != cudaSuccess) {
            set_error("ctu_filter_components: memset: %s", cudaGetErrorString(e));
            return (int)e;
        }
        if (vec) ccl_select_kernel<true><<<chunks, kCclThreads, 0, st>>>(ws.parent, ws.size, V, cpv, ws.best);
        else ccl_select_kernel<false><<<chunks, kCclThreads, 0, st>>>(ws.parent, ws.size, V, cpv, ws.best);
    }
    if (in_dtype == CTU_MASK_U8) {
        const unsigned char* i8 = (const unsigned char*)in;
        unsigned char* o8 = (unsigned char*)out;
        if (vec) ccl_filter_kernel<unsigned char, true><<<chunks, kCclThreads, 0, st>>>(i8, o8, ws.parent, ws.size, ws.best, min_size, V, cpv);
        else ccl_filter_kernel<unsigned char, false><<<chunks, kCclThreads, 0, st>>>(i8, o8, ws.parent, ws.size, ws.best, min_size, V, cpv);
    } else {
        const float* i32 = (const float*)in;
        float* o32 = (float*)out;
        if (vec) ccl_filter_kernel<float, true><<<chunks, kCclThreads, 0, st>>>(i32, o32, ws.parent, ws.size, ws.best, min_size, V, cpv);
        else ccl_filter_kernel<float, false><<<chunks, kCclThreads, 0, st>>>(i32, o32, ws.parent, ws.size, ws.best, min_size, V, cpv);
    }
    return check_launch("ctu_filter_components");
}
