// Dropout3d keep factors (nn.Dropout3d at models.py:34,46,97,411,438,492 of the reference).
// Dropout3d on a 5-D tensor multiplies channel c of sample n by k[n][c] in {0, 1/(1-p)}: a handful of numbers per site,
// which the BatchNorm+ReLU(+MaxPool) kernels that precede every dropout site apply in their epilogue (bn.cu).
// One launch draws the factors of every site of a pass from a counter-based Philox4x32-10, counter = (pass, site,
// sample*cpad + channel), key = the caller's 64-bit seed.  The pass number lives in device memory and the same launch
// advances it, so a captured CUDA graph draws fresh masks on every replay; the launch is a single block, so every thread
// reads the pass number before the barrier behind which thread 0 writes the next one.
#include "common.cuh"

namespace ctu {

constexpr int kDropThreads = 256;

struct DropSites {
    int nsite;
    int site[CTU_DROPOUT_MAX_SITES];
    int c[CTU_DROPOUT_MAX_SITES];
    int cpad[CTU_DROPOUT_MAX_SITES];
    long long off[CTU_DROPOUT_MAX_SITES + 1];   // first factor of each site in `keep`; off[nsite] = total
    float p[CTU_DROPOUT_MAX_SITES];
};

__global__ void __launch_bounds__(kDropThreads) dropout3d_keep_kernel(DropSites s, unsigned long long key,
                                                                      unsigned long long* pass_counter,
                                                                      float* __restrict__ keep) {
    const unsigned long long pass = pass_counter != nullptr ? *pass_counter : 0ull;
    __syncthreads();
    if (threadIdx.x == 0 && pass_counter != nullptr) *pass_counter = pass + 1;
    int si = 0;
    for (long long i = threadIdx.x; i < s.off[s.nsite]; i += kDropThreads) {
        while (i >= s.off[si + 1]) ++si;                 // i only grows: the site index follows it
        const long long local = i - s.off[si];
        const int ch = (int)(local % s.cpad[si]);
        const float p = s.p[si];
        float k = 0.f;                                   // pad lanes and p == 1: zero
        if (ch < s.c[si] && p < 1.f) {
            uint32_t r[4] = {(uint32_t)pass, (uint32_t)(pass >> 32), (uint32_t)s.site[si], (uint32_t)local};
            philox4x32_10(r, (uint32_t)key, (uint32_t)(key >> 32));
            const float u = (float)(r[0] >> 8) * (1.f / 16777216.f);     // uniform [0, 1), 24 bits
            k = u >= p ? 1.f / (1.f - p) : 0.f;          // kept with probability 1 - p
        }
        keep[i] = k;
    }
}

}  // namespace ctu

using namespace ctu;

extern "C" int ctu_dropout3d_keep(int nsite, const int* h_site, const int* h_channels, const float* h_p, int n,
                                  unsigned long long seed, unsigned long long* pass_counter, float* keep,
                                  ctu_stream stream) {
    CTU_REQUIRE(nsite >= 1 && nsite <= CTU_DROPOUT_MAX_SITES && h_site && h_channels && h_p && n > 0 && keep,
                "ctu_dropout3d_keep: bad arguments (nsite=%d)", nsite);
    DropSites s = {};
    s.nsite = nsite;
    long long off = 0;
    for (int i = 0; i < nsite; ++i) {
        CTU_REQUIRE(h_channels[i] > 0 && h_site[i] >= 0 && h_p[i] >= 0.f && h_p[i] <= 1.f,
                    "ctu_dropout3d_keep: site %d: channels %d, id %d, p %g", i, h_channels[i], h_site[i], (double)h_p[i]);
        s.site[i] = h_site[i];
        s.c[i] = h_channels[i];
        s.cpad[i] = (h_channels[i] + 7) / 8 * 8;
        s.p[i] = h_p[i];
        s.off[i] = off;
        off += (long long)n * s.cpad[i];
    }
    s.off[nsite] = off;
    dropout3d_keep_kernel<<<1, kDropThreads, 0, (cudaStream_t)stream>>>(s, seed, pass_counter, keep);
    return check_launch("ctu_dropout3d_keep");
}
