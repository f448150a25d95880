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
