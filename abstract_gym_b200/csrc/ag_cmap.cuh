// ag_cmap.cuh -- the configuration-space map: its layout and the readers' side (k_rollout_lut, k_check_motion,
// k_cspace).  The producer (k_cspace_build) and the library's cache of maps are in ag_cmap.cu.
//
// 2^CB1 x 2^CB2 bins over (joint_1, joint_2) mod 2pi, one bit each.  The bin of a pose with |q| < 2^20 comes from the
// joint phases x = low word of fma(q, 2^32/2pi, PHASE_MAGIC): bit ((x1 >> (32 - CB1)) << CB2) | (x2 >> (32 - CB2)) of
// the map, word bit >> 5.  CLEAR: no pose of the bin collides or reaches the target (k_cspace_build); SET: evaluate.
#pragma once
#include "ag_device.cuh"

#ifndef AG_CMAP_B1
#define AG_CMAP_B1 10
#endif
#ifndef AG_CMAP_B2
#define AG_CMAP_B2 8
#endif

namespace agd {

constexpr int CB1 = AG_CMAP_B1, CB2 = AG_CMAP_B2;
static_assert(CB1 >= 6 && CB2 >= 6 && CB1 + CB2 <= 20, "the map must fit shared memory");
constexpr int CMAP_WORDS = 1 << (CB1 + CB2 - 5);
constexpr double PHASE_MAGIC = 6755399441055744.0;       // 1.5 * 2^52: the add rounds to an integer in the low word
constexpr double TWO_PI = 6.283185307179586476925;
constexpr double PHASE_SCALE = 4294967296.0 / TWO_PI;    // phase units (2^-32 turn) per radian

__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}

// the phase word of one angle: q mod 2pi as a 32-bit turn fraction, right for |q| < 2^20 (cmap_in_range) only.
// k_rollout_lut passes the scale as a kernel parameter, which keeps the constant out of its hot loop's registers.
__device__ __forceinline__ uint32_t cmap_phase(double q, double scale = PHASE_SCALE) {
    return (uint32_t)__double2loint(fma(q, scale, PHASE_MAGIC));
}

// the range of the phase: below 2^20 the fma stays in [2^52, 2^53) on both sides of 0.  NaN is out of range.
__device__ __forceinline__ bool cmap_in_range(double q) { return fabs(q) < 1048576.0; }

// the bit of the bin of phases (x1, x2) in the map at shared-window address cmap_a
__device__ __forceinline__ bool cmap_bit(uint32_t cmap_a, uint32_t x1, uint32_t x2) {
    const uint32_t bit = ((x1 >> (32 - CB1)) << CB2) | (x2 >> (32 - CB2));
    return ((lds_u32(cmap_a + ((bit >> 3) & ~3u)) >> (bit & 31u)) & 1u) != 0u;
}

// true: pose (q1, q2) needs the full check -- its bin is SET, or an angle is outside the phase's range (or NaN).
// false: the pose certainly neither collides nor reaches the target.
__device__ __forceinline__ bool cmap_needs_check(uint32_t cmap_a, double q1, double q2) {
    return cmap_bit(cmap_a, cmap_phase(q1), cmap_phase(q2)) || !cmap_in_range(q1) || !cmap_in_range(q2);
}

// the map words (global memory) -> dst in shared memory; every thread of the block calls it, `stride` = block size
__device__ __forceinline__ void cmap_to_shared(unsigned char *dst, const uint32_t *map, int stride) {
    const uint4 *src = reinterpret_cast<const uint4 *>(map);
    for (int i = threadIdx.x; i < CMAP_WORDS / 4; i += stride) reinterpret_cast<uint4 *>(dst)[i] = src[i];
}

// The directions in which link 1 (origin -> length l1) meets the closed box X0..X1 x Y0..Y1 (an inflated square): the
// angular extent of box n (disc of radius l1) seen from the origin.  That set is convex and, unless the origin lies inside
// the box, does not contain the origin, so its extent is spanned by its vertices: corners inside the disc and circle /
// edge crossings (a ray from the centre is never tangent to the circle).  half < 0: never; half >= pi: always.
static __device__ void hazard_interval(double X0, double Y0, double X1, double Y1, double l1, float &mid, float &half) {
    if (X0 <= 0.0 && X1 >= 0.0 && Y0 <= 0.0 && Y1 >= 0.0) { mid = 0.0f; half = 4.0f; return; }
    const double r2 = l1 * l1;
    const double ref = atan2(0.5 * (Y0 + Y1), 0.5 * (X0 + X1));
    double lo = 1.0e9, hi = -1.0e9;
    auto take = [&](double px, double py) {
        double a = atan2(py, px) - ref;
        a -= TWO_PI * rint(a / TWO_PI);
        lo = fmin(lo, a); hi = fmax(hi, a);
    };
    const double XS[2] = {X0, X1}, YS[2] = {Y0, Y1};
    for (int i = 0; i < 2; ++i)
        for (int j = 0; j < 2; ++j)
            if (XS[i] * XS[i] + YS[j] * YS[j] <= r2) take(XS[i], YS[j]);
    for (int i = 0; i < 2; ++i) {
        if (fabs(XS[i]) <= l1) {
            const double y = sqrt(r2 - XS[i] * XS[i]);
            if (y >= Y0 && y <= Y1) take(XS[i], y);
            if (-y >= Y0 && -y <= Y1) take(XS[i], -y);
        }
        if (fabs(YS[i]) <= l1) {
            const double xx = sqrt(r2 - YS[i] * YS[i]);
            if (xx >= X0 && xx <= X1) take(xx, YS[i]);
            if (-xx >= X0 && -xx <= X1) take(-xx, YS[i]);
        }
    }
    if (hi < lo) { mid = 0.0f; half = -1.0f; return; }
    mid = (float)(ref + 0.5 * (lo + hi));
    half = (float)(0.5 * (hi - lo));
}

}  // namespace agd

// The map for one launch whose staged grid takes `smem` bytes of dynamic shared memory.
struct CmapLaunch {
    const uint32_t *map;   // the map words in global memory; nullptr: the launch takes its general form
    uint32_t off;          // byte offset of the map's shared-memory copy in the dynamic segment
    size_t smem;           // dynamic shared memory of the launch, the map included
};

// cspace_map_applies: the grid is one staged grid with an obstacle list (S <= 32, at most AG_LIST_MAX occupied cells by
// ag_grid.max_occupied), the only grids the map is built for.
bool cspace_map_applies(const agd::GridDev &G, int32_t max_occupied);
// cspace_map_for_launch: where the map applies, the library's cached map of this grid and these parameters, after
// enqueuing on `s` the k_cspace_build launch that checks it against the grid's current content on the device (and
// rebuilds it if it differs).  out->map = nullptr when the map does not apply or no cache entry can be had (inside a
// stream capture before the grid's first uncaptured launch, or an allocation failure): the caller then takes its
// general form, whose results are identical.
ag_status cspace_map_for_launch(const ag_params &P, const agd::GridDev &G, int32_t max_occupied, size_t smem, cudaStream_t s,
                                CmapLaunch *out);
