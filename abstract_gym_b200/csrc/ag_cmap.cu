// ag_cmap.cu -- the configuration-space map (layout: ag_cmap.cuh): k_cspace_build, which makes it, the library's cache of
// maps, which hands one to each launch that reads it (cspace_map_for_launch), and ag_cspace_map, which builds one into a
// caller's buffer.  DESIGN.md "K4, scene_0 class".
#include <atomic>
#include <cstring>
#include <mutex>

#include "ag_cmap.cuh"
#include "ag_rollout.cuh"

using namespace agd;

namespace {

constexpr int CMAP_HDR_WORDS = 64;                       // 256-byte header in front of the map words
constexpr int CMAP_SLOTS = 16;
struct CmapHeader {
    unsigned long long key;                              // hash of everything the map depends on; 0 = never built
    unsigned int done[CMAP_SLOTS];                       // blocks finished, one counter per in-flight build
};
static_assert(sizeof(CmapHeader) <= CMAP_HDR_WORDS * 4, "header");

// One bit per bin of (joint_1, joint_2) mod 2pi: CLEAR = for every pose of the bin both links stay farther than CMAP_MG
// from every occupied square and the end effector stays outside the target box (scene_0.py:129-130) by more than
// CMAP_MG, i.e. the step is certainly uneventful and the hot loop needs no forward kinematics at all -- two DFMA for
// the phases, one shared-memory word, one bit test.  SET = "look closer": the lane takes the slow path, which decides
// exactly as before.  So the map only has to be CONSERVATIVE; it is built from lower bounds of distances:
//   * over a bin, joint_1 in [a1-d1, a1+d1] and joint_2 in [a2-d2, a2+d2], the elbow stays within the sagitta
//     l1(1-cos d1) of the chord Ea..Eb and link 2's direction vector within l2(1-cos d2) of the triangle 0, Ua, Ub, so
//     link 2 sweeps a subset of the convex polygon hull({Ea,Eb} + {0,Ua,Ub}) inflated by the two sagittas;
//   * the distance from that polygon to a square is bounded from below by the largest separation along a finite set
//     of unit axes (every axis gives a valid lower bound; the set -- box normals, the link normals at the bin's centre
//     and edges, the chord normal, and the directions from the square's corners to the centre pose's elbow and end
//     effector -- makes the bound tight for edge/vertex and vertex/vertex contacts);
//   * link 1 depends on joint_1 only and uses the exact angular intervals of hazard_interval().
// 2.0e-6 m covers the rounding of the phase (< 1e-9 rad), of this float64 construction, and the reference's own
// rounding noise (< 1e-12 m): the same margin the float32 broad phase uses.
// The map depends on the grid, the link lengths, the target and its tolerance.  It lives in a library-owned device
// buffer that is reused between launches: every launch re-derives a 64-bit key from the CURRENT grid words and
// parameters on the device (thread 0 of each block, ~100 words) and rebuilds the map only when the stored key differs.
constexpr double CMAP_MG = 2.0e-6;
constexpr int CMAP_BUILD_BLOCKS = 128;
constexpr uint32_t CMAP_VERSION = 1;

struct V2 { double x, y; };

__device__ __forceinline__ unsigned long long mix64(unsigned long long h, unsigned long long v) {
    h ^= v;
    h *= 0x100000001B3ull;                                                       // FNV-1a over 64-bit words
    return h ^ (h >> 29);
}

// separation of the point set P and the box (centre c, half extents hx, hy) along the unit axis n (negative: overlap)
template <int NP>
__device__ __forceinline__ double axis_gap(V2 n, const V2 (&P)[NP], V2 c, double hx, double hy) {
    double lo = 1.0e300, hi = -1.0e300;
#pragma unroll
    for (int i = 0; i < NP; ++i) {
        const double d = n.x * P[i].x + n.y * P[i].y;
        lo = fmin(lo, d); hi = fmax(hi, d);
    }
    const double cc = n.x * c.x + n.y * c.y, r = fabs(n.x) * hx + fabs(n.y) * hy;
    return fmax(lo - (cc + r), (cc - r) - hi);
}

__global__ void __launch_bounds__(256)
k_cspace_build(const __grid_constant__ ag_params P, const __grid_constant__ GridDev G, uint32_t *buf, uint32_t slot) {
    __shared__ unsigned long long s_key;
    __shared__ int s_skip, s_m;
    __shared__ double s_sq[AG_LIST_MAX][4];
    __shared__ float s_hz[2 * AG_LIST_MAX];
    CmapHeader *H = reinterpret_cast<CmapHeader *>(buf);
    if (threadIdx.x == 0) {
        unsigned long long h = 0xCBF29CE484222325ull;
        h = mix64(h, ((unsigned long long)CMAP_VERSION << 48) | ((unsigned long long)CB1 << 40) | ((unsigned long long)CB2 << 32) | (unsigned)G.S);
        const double par[6] = {P.link_1, P.link_2, P.target_x, P.target_y, P.reach_eps, G.side};
        for (int i = 0; i < 6; ++i) h = mix64(h, (unsigned long long)__double_as_longlong(par[i]));
        int m = 0;
        for (int r = 0; r < G.S; ++r) {
            h = mix64(h, (unsigned long long)__double_as_longlong(G.min_y[r]));
            h = mix64(h, (unsigned long long)__double_as_longlong(G.min_x[r]));
            for (int w = 0; w < G.wpr; ++w) {
                uint32_t word = G.bits[r * G.wpr + w];
                h = mix64(h, word);
                while (word) {
                    const int c = (w << 5) + __ffs(word) - 1;
                    word &= word - 1;
                    if (m < AG_LIST_MAX && c < G.S) {
                        const double mnx = G.min_x[c], mny = G.min_y[r];
                        s_sq[m][0] = mnx; s_sq[m][1] = mny;
                        s_sq[m][2] = __dadd_rn(mnx, G.side); s_sq[m][3] = __dadd_rn(mny, G.side);   // occupancy_grid.py:66-67
                    }
                    ++m;
                }
            }
        }
        h |= 1ull;                                                               // 0 means "never built"
        s_key = h;
        s_m = m > AG_LIST_MAX ? -1 : m;                                          // no obstacle list: every bin is slow
        s_skip = (*reinterpret_cast<volatile unsigned long long *>(&H->key) == h) ? 1 : 0;
    }
    __syncthreads();
    if (!s_skip) {
        const int m = s_m;
        if ((int)threadIdx.x < m)
            hazard_interval(s_sq[threadIdx.x][0] - CMAP_MG, s_sq[threadIdx.x][1] - CMAP_MG, s_sq[threadIdx.x][2] + CMAP_MG,
                            s_sq[threadIdx.x][3] + CMAP_MG, P.link_1, s_hz[2 * threadIdx.x], s_hz[2 * threadIdx.x + 1]);
        __syncthreads();
        constexpr int N1c = 1 << CB1, N2c = 1 << CB2;
        const double l1 = P.link_1, l2 = P.link_2;
        double sd, cd;
        sincospi(1.0 / (double)N1c, &sd, &cd);
        const double sag1 = l1 * (1.0 - cd);
        sincospi(1.0 / (double)N2c, &sd, &cd);
        const double sag2 = l2 * (1.0 - cd);
        const double infl = sag1 + sag2 + CMAP_MG;
        const float hw1 = (float)(TWO_PI / (double)(2 * N1c)) + 2.0e-6f;          // half a bin of joint_1 + rounding
        for (int bin = blockIdx.x * 256 + threadIdx.x; bin < N1c * N2c; bin += gridDim.x * 256) {   // a warp = 32 bins of joint_2
            const int b1 = bin >> CB2, b2 = bin & (N2c - 1);
            bool haz = m < 0;
            // ---- link 1: exact angular intervals
            const float th1 = ((float)b1 + 0.5f) * (float)(TWO_PI / (double)N1c);
            for (int k = 0; k < m; ++k) {
                float dlt = th1 - s_hz[2 * k];
                dlt -= (float)TWO_PI * rintf(dlt * (float)(1.0 / TWO_PI));
                if (fabsf(dlt) <= s_hz[2 * k + 1] + hw1) haz = true;
            }
            // ---- link 2: the swept polygon against every square
            V2 Ea, Eb, Ec, Ua, Ub, Uc;
            sincospi(2.0 * (double)b1 / (double)N1c, &Ea.y, &Ea.x);
            sincospi(2.0 * (double)(b1 + 1) / (double)N1c, &Eb.y, &Eb.x);
            sincospi((2.0 * (double)b1 + 1.0) / (double)N1c, &Ec.y, &Ec.x);
            sincospi(2.0 * (double)b2 / (double)N2c, &Ua.y, &Ua.x);
            sincospi(2.0 * (double)(b2 + 1) / (double)N2c, &Ub.y, &Ub.x);
            sincospi((2.0 * (double)b2 + 1.0) / (double)N2c, &Uc.y, &Uc.x);
            const V2 n1c = {Ec.x, Ec.y};                                          // normal of the elbow chord = link 1's direction
            const V2 n2a = {-Ua.y, Ua.x}, n2b = {-Ub.y, Ub.x}, n2c = {-Uc.y, Uc.x};   // link 2's normals at the bin's edges / centre
            const V2 ea = {l1 * Ea.x, l1 * Ea.y}, eb = {l1 * Eb.x, l1 * Eb.y}, ec = {l1 * Ec.x, l1 * Ec.y};
            const V2 ua = {l2 * Ua.x, l2 * Ua.y}, ub = {l2 * Ub.x, l2 * Ub.y};
            const V2 gc = {ec.x + l2 * Uc.x, ec.y + l2 * Uc.y};
            const V2 poly[6] = {ea, eb, {ea.x + ua.x, ea.y + ua.y}, {ea.x + ub.x, ea.y + ub.y},
                                {eb.x + ua.x, eb.y + ua.y}, {eb.x + ub.x, eb.y + ub.y}};
            for (int k = 0; k < m && !haz; ++k) {
                const V2 c = {0.5 * (s_sq[k][0] + s_sq[k][2]), 0.5 * (s_sq[k][1] + s_sq[k][3])};
                const double hx = 0.5 * (s_sq[k][2] - s_sq[k][0]), hy = 0.5 * (s_sq[k][3] - s_sq[k][1]);
                double gap = axis_gap(V2{1.0, 0.0}, poly, c, hx, hy);
                gap = fmax(gap, axis_gap(V2{0.0, 1.0}, poly, c, hx, hy));
                gap = fmax(gap, axis_gap(n2c, poly, c, hx, hy));
                gap = fmax(gap, axis_gap(n2a, poly, c, hx, hy));
                gap = fmax(gap, axis_gap(n2b, poly, c, hx, hy));
                gap = fmax(gap, axis_gap(n1c, poly, c, hx, hy));
#pragma unroll 1
                for (int j = 0; j < 8; ++j) {                                     // corner -> centre pose's end effector / elbow
                    const double qx = (j & 1) ? s_sq[k][2] : s_sq[k][0], qy = (j & 2) ? s_sq[k][3] : s_sq[k][1];
                    const V2 from = (j & 4) ? ec : gc;
                    const double vx = from.x - qx, vy = from.y - qy, nv = sqrt(vx * vx + vy * vy);
                    if (nv > 1.0e-9) gap = fmax(gap, axis_gap(V2{vx / nv, vy / nv}, poly, c, hx, hy) * (1.0 - 1.0e-12));
                }
                if (!(gap > infl)) haz = true;
            }
            // ---- the target box (scene_0.py:129-130) against the box of the swept end effector
            {
                const double gx0 = fmin(fmin(poly[2].x, poly[3].x), fmin(poly[4].x, poly[5].x)) - infl;
                const double gx1 = fmax(fmax(poly[2].x, poly[3].x), fmax(poly[4].x, poly[5].x)) + infl;
                const double gy0 = fmin(fmin(poly[2].y, poly[3].y), fmin(poly[4].y, poly[5].y)) - infl;
                const double gy1 = fmax(fmax(poly[2].y, poly[3].y), fmax(poly[4].y, poly[5].y)) + infl;
                const double e = fabs(P.reach_eps);
                if (!(gx0 > P.target_x + e || gx1 < P.target_x - e || gy0 > P.target_y + e || gy1 < P.target_y - e)) haz = true;
            }
            const uint32_t word = __ballot_sync(0xFFFFFFFFu, haz);
            if ((threadIdx.x & 31) == 0) buf[CMAP_HDR_WORDS + (bin >> 5)] = word;
        }
    }
    // the last block of this launch publishes the key (blocks that skipped count too: the map they saw was complete)
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        if (atomicAdd(&H->done[slot], 1u) == gridDim.x - 1) {
            H->done[slot] = 0;
            *reinterpret_cast<volatile unsigned long long *>(&H->key) = s_key;
            __threadfence();
        }
    }
}

// ---- the library-owned buffers of the configuration-space maps: up to 32 entries (33 KB each) per process, found by (device, grid
// pointers, parameters); the CONTENT is validated on the device by every launch (k_cspace_build), so a grid that was
// rewritten in place, or a new grid at a recycled address, just rebuilds the entry.
struct CmapEntry {
    int dev = -1;
    const void *bits = nullptr, *min_x = nullptr;
    double par[6] = {0, 0, 0, 0, 0, 0};
    int S = 0;
    uint32_t *buf = nullptr;
    unsigned long long last_use = 0;
};
constexpr int CMAP_ENTRIES = 32;
std::mutex g_cmap_mutex;
CmapEntry g_cmap[CMAP_ENTRIES];
unsigned long long g_cmap_clock = 0;

// the entry's device buffer (header + map), or nullptr when the map form cannot be used for this launch
uint32_t *cmap_buffer(const ag_params &P, const GridDev &G, cudaStream_t s) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(s, &cap) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    const bool capturing = cap != cudaStreamCaptureStatusNone;
    const double par[6] = {P.link_1, P.link_2, P.target_x, P.target_y, P.reach_eps, G.side};
    std::lock_guard<std::mutex> lock(g_cmap_mutex);
    CmapEntry *hit = nullptr, *lru = &g_cmap[0];
    for (CmapEntry &e : g_cmap) {
        if (e.buf != nullptr && e.dev == dev && e.bits == G.bits && e.min_x == G.min_x && e.S == G.S &&
            std::memcmp(e.par, par, sizeof(par)) == 0) { hit = &e; break; }
        if (e.last_use < lru->last_use) lru = &e;
    }
    if (hit == nullptr) {
        if (capturing) return nullptr;                        // no allocation / synchronisation inside a stream capture
        if (lru->buf != nullptr) {
            // the buffer changes hands: launches that still read the old map (any stream of its device) must be done
            int cur = dev;
            if (lru->dev != cur && cudaSetDevice(lru->dev) != cudaSuccess) return nullptr;
            cudaDeviceSynchronize();
            if (lru->dev != cur) { cudaFree(lru->buf); lru->buf = nullptr; cudaSetDevice(cur); }
        }
        if (lru->buf == nullptr && cudaMalloc(&lru->buf, (size_t)(CMAP_HDR_WORDS + CMAP_WORDS) * 4) != cudaSuccess) {
            cudaGetLastError();
            lru->buf = nullptr; lru->dev = -1;
            return nullptr;
        }
        if (cudaMemsetAsync(lru->buf, 0, CMAP_HDR_WORDS * 4, s) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        lru->dev = dev; lru->bits = G.bits; lru->min_x = G.min_x; lru->S = G.S;
        std::memcpy(lru->par, par, sizeof(par));
        hit = lru;
    }
    hit->last_use = ++g_cmap_clock;
    return hit->buf;
}
}  // namespace

bool cspace_map_applies(const GridDev &G, int32_t max_occupied) {
    return G.stage && G.n_grids == 1 && G.S <= 32 && max_occupied >= 0 && max_occupied <= AG_LIST_MAX;
}

ag_status cspace_map_for_launch(const ag_params &P, const GridDev &G, int32_t max_occupied, size_t smem, cudaStream_t s,
                                CmapLaunch *out) {
    out->map = nullptr; out->off = 0; out->smem = smem;
    uint32_t *buf = cspace_map_applies(G, max_occupied) ? cmap_buffer(P, G, s) : nullptr;
    if (buf == nullptr) return AG_OK;
    static std::atomic<unsigned> next_build{0};
    k_cspace_build<<<CMAP_BUILD_BLOCKS, 256, 0, s>>>(P, G, buf, next_build.fetch_add(1, std::memory_order_relaxed) % CMAP_SLOTS);
    const ag_status st = launched();
    if (st != AG_OK) return st;
    out->map = buf + CMAP_HDR_WORDS;
    out->off = (uint32_t)((smem + 15) & ~(size_t)15);
    out->smem = (size_t)out->off + (size_t)CMAP_WORDS * 4;
    return AG_OK;
}

extern "C" int64_t ag_cspace_map_words(int32_t *b1, int32_t *b2) {
    if (b1) *b1 = CB1;
    if (b2) *b2 = CB2;
    return CMAP_WORDS;
}

// the map alone, into the caller's buffer: built in a scratch buffer with the header in front
extern "C" ag_status ag_cspace_map(const ag_params *p, const ag_grid *g, uint32_t *map, void *stream) {
    if (!p || !g || !map) return AG_ERR_NULL;
    if (g->n_grids != 1 || g->S > 32) return AG_ERR_SHAPE;
    if ((uintptr_t)map % 16) return AG_ERR_ALIGN;
    GridDev G;
    size_t smem;
    ag_status st = make_grid_dev(p, g, 0, AG_ENGINE_FAST, &G, &smem);
    if (st) return st;
    cudaStream_t s = (cudaStream_t)stream;
    uint32_t *buf = nullptr;
    cudaError_t e = cudaMallocAsync(&buf, (size_t)(CMAP_HDR_WORDS + CMAP_WORDS) * 4, s);
    if (e != cudaSuccess) return (ag_status)e;
    e = cudaMemsetAsync(buf, 0, CMAP_HDR_WORDS * 4, s);
    if (e == cudaSuccess) {
        k_cspace_build<<<CMAP_BUILD_BLOCKS, 256, 0, s>>>(*p, G, buf, 0);
        e = (cudaError_t)launched();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(map, buf + CMAP_HDR_WORDS, (size_t)CMAP_WORDS * 4, cudaMemcpyDeviceToDevice, s);
    cudaFreeAsync(buf, s);
    return (ag_status)e;
}
