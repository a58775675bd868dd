// Defect regions: connected components of a label map (8-connectivity, per nonzero class) with canonical ids and
// per-region class, area, box and mean uncertainty.  See include/uaps_b200.h for the contract and DESIGN.md f10.
//
// Block-based union-find (Playne & Hawick 2018), working in per-image raster indices p = y * W + x:
//   1. local:   one CTA per 32x32 tile labels it in shared memory; a union always links the larger root under the
//               smaller one (atomicMin), so every root is the smallest raster index of its set.  Each pixel's tile-local
//               root goes to `regions`, which serves as the global parent array; background is -1.
//   2. border:  one thread per tile-border pixel unites it with its backward neighbours in other tiles, on the global
//               parent array, with the same min-linking union.  A component's root is then its first raster pixel.
//   3. flatten: every pixel's parent becomes its root; per fixed raster chunk of each image the roots are counted.
//   4. scan:    one CTA per image folds the chunk counts in chunk order (exclusive offsets, the image's region count)
//               and initialises the image's rows of the stats table.
//   5. ids:     roots get id = 1 + (roots before them in raster order): chunk offset + block scan of the chunk's root
//               flags.  A root's slot holds -id - 1 until step 6 rewrites it.
//   6. relabel: every pixel reads its root's id; area and box by integer atomics and the uncertainty sum by fp64 atomics,
//               aggregated per warp over the lanes that share a region id first.
//   7. means:   unc_mean = sum / area in fp64, rounded once to fp32 (only with an uncertainty map).
// The ids depend on the components only, never on scheduling, so the map, ids and integer statistics are bitwise
// reproducible.  Every launch writes what later launches read and the launch sequence depends on the arguments only:
// no initialised workspace, no host synchronisation, graph-capturable.
#include "common.cuh"
#include <climits>
#include <cooperative_groups.h>
#include <cooperative_groups/reduce.h>

namespace uaps {
namespace rgn {
namespace cg = cooperative_groups;

constexpr int TILE = 32;                    // local step: TILE x TILE pixels per CTA, one per thread
constexpr int THREADS = 256;                // chunked steps
constexpr int ROUNDS = 8;
constexpr int CHUNK = THREADS * ROUNDS;     // pixels of one image per CTA in steps 3, 5 and 6
constexpr int BORDER_THREADS = 3 * TILE - 2;
constexpr int BG = -1;

static_assert(sizeof(UapsRegion) == 32, "UapsRegion is 8 words");

__device__ __forceinline__ int ld_parent(const int* P, int x) { return __ldcg(P + x); }

// ---- union-find on a shared tile ------------------------------------------------------------------------------------
__device__ __forceinline__ int find_s(const volatile int* par, int x) {
    int p;
    while ((p = par[x]) != x) x = p;
    return x;
}
__device__ __forceinline__ void unite_s(int* par, int a, int b) {
    while (true) {
        a = find_s(par, a);
        b = find_s(par, b);
        if (a == b) return;
        if (a > b) { const int t = a; a = b; b = t; }
        const int old = atomicMin(par + b, a);
        if (old == b) return;
        b = old;                            // b was linked meanwhile: unite a with where it went
    }
}

// ---- union-find on the global parent array (one image) -------------------------------------------------------------
// Path halving: a visited node is pointed at its grandparent.  Ancestors have strictly smaller indices, so atomicMin
// keeps whichever of two racing writes is nearer the root -- a plain store could put back a farther ancestor over the
// root another thread has just written (step 3).  A root is never written.  It bounds the chains a serpentine across
// many tiles would build.
__device__ __forceinline__ int find_g(int* P, int x) {
    while (true) {
        const int p = ld_parent(P, x);
        if (p == x) return x;
        const int gp = ld_parent(P, p);
        if (gp == p) return p;
        atomicMin(P + x, gp);
        x = gp;
    }
}
__device__ __forceinline__ void unite_g(int* P, int a, int b) {
    while (true) {
        a = find_g(P, a);
        b = find_g(P, b);
        if (a == b) return;
        if (a > b) { const int t = a; a = b; b = t; }
        const int old = atomicMin(P + b, a);
        if (old == b) return;
        b = old;
    }
}

struct Geo {
    int H, W;
    unsigned tiles_x;
    long long HW;
    unsigned chunks;                        // per image
};

// 1. tile-local labelling
__global__ void __launch_bounds__(TILE * TILE) regions_local_kernel(const uint8_t* __restrict__ labels, int* __restrict__ regions,
                                                                    const Geo g) {
    __shared__ int par[TILE * TILE];
    __shared__ uint8_t lab[TILE * TILE];
    grid_dep_wait();
    const unsigned b = blockIdx.y;
    const unsigned tx0 = (blockIdx.x % g.tiles_x) * TILE, ty0 = (blockIdx.x / g.tiles_x) * TILE;
    const int lx = threadIdx.x, ly = threadIdx.y, l = ly * TILE + lx;
    const bool in = tx0 + lx < (unsigned)g.W && ty0 + ly < (unsigned)g.H;
    const long long p = in ? (long long)(ty0 + ly) * g.W + (tx0 + lx) : 0;
    const uint8_t c = in ? labels[(size_t)b * g.HW + p] : 0;
    // one warp per tile row: each pixel starts linked to the first pixel of its horizontal run (same class, contiguous)
    const uint8_t cl = __shfl_up_sync(0xffffffffu, c, 1), cr = __shfl_down_sync(0xffffffffu, c, 1);
    const bool same_left = c != 0 && lx > 0 && cl == c, same_right = c != 0 && lx < TILE - 1 && cr == c;
    const unsigned starts = __ballot_sync(0xffffffffu, c != 0 && !same_left);
    const unsigned upto = lx == TILE - 1 ? 0xffffffffu : (2u << lx) - 1u;
    lab[l] = c;
    par[l] = ly * TILE + (31 - __clz(starts & upto));
    __syncthreads();
    // a run meets each run of the row above once: where an overlap with it begins, or diagonally at its two ends
    if (c != 0 && ly > 0) {
        const uint8_t up = lab[l - TILE];
        const uint8_t ul = lx > 0 ? lab[l - TILE - 1] : 0, ur = lx < TILE - 1 ? lab[l - TILE + 1] : 0;
        if (up == c && (!same_left || ul != c)) unite_s(par, l, l - TILE);
        if (up != c && !same_left && ul == c) unite_s(par, l, l - TILE - 1);
        if (up != c && !same_right && ur == c) unite_s(par, l, l - TILE + 1);
    }
    __syncthreads();
    if (in) {
        int v = BG;
        if (c != 0) {
            const int r = find_s(par, l);
            v = (int)((long long)(ty0 + r / TILE) * g.W + (tx0 + r % TILE));
        }
        regions[(size_t)b * g.HW + p] = v;
    }
}

// 2. unions across tile borders: top row (up-left, up, up-right; and left at the tile's corner), left column below
//    the top row (left, up-left), right column below the top row (up-right).  Every pair of 8-neighbours in different
//    tiles is visited once, from its later pixel.
__global__ void __launch_bounds__(128) regions_border_kernel(const uint8_t* __restrict__ labels, int* __restrict__ regions,
                                                             const Geo g) {
    grid_dep_wait();
    const unsigned b = blockIdx.y;
    const unsigned tx0 = (blockIdx.x % g.tiles_x) * TILE, ty0 = (blockIdx.x / g.tiles_x) * TILE;
    const int t = threadIdx.x;
    if (t >= BORDER_THREADS) return;
    unsigned x, y;
    if (t < TILE) { x = tx0 + t; y = ty0; }
    else if (t < 2 * TILE - 1) { x = tx0; y = ty0 + 1 + (t - TILE); }
    else { x = tx0 + TILE - 1; y = ty0 + 1 + (t - (2 * TILE - 1)); }
    if (x >= (unsigned)g.W || y >= (unsigned)g.H) return;
    const uint8_t* L = labels + (size_t)b * g.HW;
    int* P = regions + (size_t)b * g.HW;
    const int W = g.W;
    const int p = (int)((long long)y * W + x);
    const uint8_t c = L[p];
    if (c == 0) return;
    const bool top = t < TILE, left = t == 0 || (t >= TILE && t < 2 * TILE - 1);
    const bool right = t == TILE - 1 || t >= 2 * TILE - 1;
    if (left && x > 0) {
        if (L[p - 1] == c) unite_g(P, p, p - 1);
        if (y > 0 && L[p - W - 1] == c) unite_g(P, p, p - W - 1);
    }
    if (top && y > 0) {
        if (!left && x > 0 && L[p - W - 1] == c) unite_g(P, p, p - W - 1);
        if (L[p - W] == c) unite_g(P, p, p - W);
        if (!right && x + 1 < (unsigned)W && L[p - W + 1] == c) unite_g(P, p, p - W + 1);
    }
    if (right && y > 0 && x + 1 < (unsigned)W && L[p - W + 1] == c) unite_g(P, p, p - W + 1);
}

// 3. parent -> root for every pixel (concurrent rewrites only ever point a pixel at an ancestor), roots per chunk
__global__ void __launch_bounds__(THREADS) regions_flatten_kernel(int* __restrict__ regions, int* __restrict__ chunk_roots,
                                                                  const Geo g) {
    __shared__ int s_cnt[THREADS / kWarp];
    grid_dep_wait();
    const unsigned b = blockIdx.y;
    int* P = regions + (size_t)b * g.HW;
    const long long base = (long long)blockIdx.x * CHUNK;
    int roots = 0;
#pragma unroll 2
    for (int r = 0; r < ROUNDS; ++r) {
        const long long q = base + r * THREADS + threadIdx.x;
        if (q >= g.HW) break;
        const int p = (int)q;
        const int v = ld_parent(P, p);
        if (v == BG) continue;
        if (v == p) { ++roots; continue; }
        const int root = find_g(P, v);
        if (root != v) P[p] = root;
    }
    roots = __reduce_add_sync(0xffffffffu, roots);
    if ((threadIdx.x & 31) == 0) s_cnt[threadIdx.x >> 5] = roots;
    __syncthreads();
    if (threadIdx.x == 0) {
        int s = 0;
#pragma unroll
        for (int w = 0; w < THREADS / kWarp; ++w) s += s_cnt[w];
        chunk_roots[(size_t)b * g.chunks + blockIdx.x] = s;
    }
}

// exclusive scan over the block in thread order; returns the block total in *total
__device__ __forceinline__ int block_exclusive_scan(int v, int* s_warp, int* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int n = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += n;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    int before = 0, all = 0;
#pragma unroll
    for (int w = 0; w < THREADS / kWarp; ++w) {
        const int s = s_warp[w];
        before += w < warp ? s : 0;
        all += s;
    }
    __syncthreads();                        // s_warp is reused by the next call
    *total = all;
    return before + inc - v;
}

// 4. per image: chunk counts -> exclusive offsets (in place, chunk order), the region count, the stats rows
__global__ void __launch_bounds__(THREADS) regions_scan_kernel(int* __restrict__ chunk_roots, int* __restrict__ count,
                                                               UapsRegion* __restrict__ stats, double* __restrict__ unc_sums,
                                                               int max_regions, const Geo g) {
    __shared__ int s_warp[THREADS / kWarp];
    grid_dep_wait();
    const unsigned b = blockIdx.x;
    int* cr = chunk_roots + (size_t)b * g.chunks;
    int carry = 0;
    for (unsigned i0 = 0; i0 < g.chunks; i0 += THREADS) {
        const unsigned i = i0 + threadIdx.x;
        const int v = i < g.chunks ? cr[i] : 0;
        int total;
        const int ex = block_exclusive_scan(v, s_warp, &total);
        if (i < g.chunks) cr[i] = carry + ex;
        carry += total;
    }
    if (threadIdx.x == 0) count[b] = carry;
    for (int i = threadIdx.x; i < max_regions; i += THREADS) {
        UapsRegion s{};                     // rows past the count stay zero
        if (i < carry) { s.y0 = INT_MAX; s.x0 = INT_MAX; }
        stats[(size_t)b * max_regions + i] = s;
        if (unc_sums != nullptr) unc_sums[(size_t)b * max_regions + i] = 0.0;
    }
}

// 5. canonical ids of the roots: a root's slot becomes -id - 1
__global__ void __launch_bounds__(THREADS) regions_ids_kernel(int* __restrict__ regions, const int* __restrict__ chunk_offsets,
                                                              const Geo g) {
    __shared__ int s_warp[THREADS / kWarp];
    grid_dep_wait();
    const unsigned b = blockIdx.y;
    int* P = regions + (size_t)b * g.HW;
    const long long base = (long long)blockIdx.x * CHUNK;
    int next = chunk_offsets[(size_t)b * g.chunks + blockIdx.x] + 1;
    for (int r = 0; r < ROUNDS; ++r) {
        const long long q = base + r * THREADS + threadIdx.x;
        if (base + r * THREADS >= g.HW) break;          // uniform over the block
        const bool root = q < g.HW && P[q] == (int)q;
        int total;
        const int ex = block_exclusive_scan(root ? 1 : 0, s_warp, &total);
        if (root) P[q] = -(next + ex) - 1;
        next += total;
    }
}

// 6. ids for every pixel, class / area / box / uncertainty sum per region
__global__ void __launch_bounds__(THREADS) regions_relabel_kernel(const uint8_t* __restrict__ labels,
                                                                  const float* __restrict__ unc, int* __restrict__ regions,
                                                                  UapsRegion* __restrict__ stats, double* __restrict__ unc_sums,
                                                                  int max_regions, const Geo g) {
    grid_dep_wait();
    const unsigned b = blockIdx.y;
    int* P = regions + (size_t)b * g.HW;
    const long long base = (long long)blockIdx.x * CHUNK;
    const auto warp = cg::tiled_partition<32>(cg::this_thread_block());
    for (int r = 0; r < ROUNDS; ++r) {
        if (base + r * THREADS >= g.HW) break;          // uniform over the block
        const long long q = base + r * THREADS + threadIdx.x;
        int id = 0;
        bool root = false;
        if (q < g.HW) {
            const int v = __ldcg(P + q);
            if (v != BG) {
                if (v < 0) {                            // this pixel is its region's root
                    id = -v - 1;
                    root = true;
                } else {                                // the root's slot: -id - 1, or id once its own thread got there
                    const int w = __ldcg(P + v);
                    id = w < 0 ? -w - 1 : w;
                }
            }
            P[q] = id;
        }
        if (max_regions == 0) continue;
        const int key = id <= max_regions ? id : 0;     // 0: no stats row
        const auto grp = cg::labeled_partition(warp, key);
        if (key == 0) continue;
        UapsRegion* s = stats + (size_t)b * max_regions + (key - 1);
        const size_t gq = (size_t)b * g.HW + q;
        if (root) s->cls = labels[gq];
        const int y = (int)(q / g.W), x = (int)(q - (long long)y * g.W);
        const int ymin = cg::reduce(grp, y, cg::less<int>()), ymax = cg::reduce(grp, y, cg::greater<int>());
        const int xmin = cg::reduce(grp, x, cg::less<int>()), xmax = cg::reduce(grp, x, cg::greater<int>());
        double u = 0.0;
        if (unc != nullptr) u = cg::reduce(grp, (double)unc[gq], cg::plus<double>());
        if (grp.thread_rank() == 0) {
            atomicAdd(&s->area, (int)grp.size());
            atomicMin(&s->y0, ymin);
            atomicMin(&s->x0, xmin);
            atomicMax(&s->y1, ymax + 1);
            atomicMax(&s->x1, xmax + 1);
            if (unc != nullptr) atomicAdd(unc_sums + (s - stats), u);
        }
    }
}

// 7. mean uncertainty of every region that has a row
__global__ void __launch_bounds__(THREADS) regions_means_kernel(const int* __restrict__ count, UapsRegion* __restrict__ stats,
                                                                const double* __restrict__ unc_sums, int B, int max_regions) {
    grid_dep_wait();
    const long long i = (long long)blockIdx.x * THREADS + threadIdx.x;
    if (i >= (long long)B * max_regions) return;
    const int b = (int)(i / max_regions), k = (int)(i - (long long)b * max_regions);
    if (k >= count[b]) return;
    stats[i].unc_mean = (float)(unc_sums[i] / (double)stats[i].area);
}

inline Geo geometry(int H, int W) {
    Geo g;
    g.H = H; g.W = W;
    g.tiles_x = (unsigned)ceil_div<long long>(W, TILE);
    g.HW = (long long)H * W;
    g.chunks = (unsigned)ceil_div<long long>(g.HW, CHUNK);
    return g;
}
inline unsigned tiles(const Geo& g) { return g.tiles_x * (unsigned)ceil_div<long long>(g.H, TILE); }
inline size_t roots_bytes(int B, const Geo& g) { return ceil_div<size_t>((size_t)B * g.chunks * sizeof(int), 256) * 256; }

}  // namespace rgn
}  // namespace uaps

using namespace uaps;

UAPS_API size_t uaps_regions_workspace_bytes(int B, int H, int W, int max_regions) {
    if (B <= 0 || H <= 0 || W <= 0 || max_regions < 0 || B > 65535 || (long long)H * W >= (1LL << 31)) return 0;
    const rgn::Geo g = rgn::geometry(H, W);
    return rgn::roots_bytes(B, g) + (size_t)B * (size_t)max_regions * sizeof(double);
}

UAPS_API int uaps_regions(const uint8_t* labels, const float* uncertainty, int B, int H, int W, int32_t* regions,
                          int32_t* count, UapsRegion* stats, int max_regions, void* workspace, size_t workspace_bytes,
                          cudaStream_t stream) {
    if (labels == nullptr || regions == nullptr || count == nullptr || workspace == nullptr) return UAPS_EINVAL;
    if (B <= 0 || H <= 0 || W <= 0 || max_regions < 0) return UAPS_EINVAL;
    if ((stats == nullptr) != (max_regions == 0)) return UAPS_EINVAL;
    if (B > 65535 || (long long)H * W >= (1LL << 31)) return UAPS_ERANGE;
    if ((uncertainty != nullptr && !aligned_to(uncertainty, 4)) || !aligned_to(regions, 4) || !aligned_to(count, 4) ||
        (stats != nullptr && !aligned_to(stats, 4)) || !aligned_to(workspace, 8))
        return UAPS_EALIGN;
    if (workspace_bytes < uaps_regions_workspace_bytes(B, H, W, max_regions)) return UAPS_EINVAL;

    const rgn::Geo g = rgn::geometry(H, W);
    int* chunk_roots = reinterpret_cast<int*>(workspace);
    double* unc_sums = (uncertainty != nullptr && max_regions > 0)
                           ? reinterpret_cast<double*>(reinterpret_cast<char*>(workspace) + rgn::roots_bytes(B, g))
                           : nullptr;
    const dim3 tile_grid(rgn::tiles(g), B), chunk_grid(g.chunks, B);
    UAPS_LAUNCH(rgn::regions_local_kernel, tile_grid, dim3(rgn::TILE, rgn::TILE), 0, stream, labels, regions, g);
    UAPS_LAUNCH(rgn::regions_border_kernel, tile_grid, dim3(128), 0, stream, labels, regions, g);
    UAPS_LAUNCH(rgn::regions_flatten_kernel, chunk_grid, dim3(rgn::THREADS), 0, stream, regions, chunk_roots, g);
    UAPS_LAUNCH(rgn::regions_scan_kernel, dim3(B), dim3(rgn::THREADS), 0, stream, chunk_roots, (int*)count, stats, unc_sums,
                max_regions, g);
    UAPS_LAUNCH(rgn::regions_ids_kernel, chunk_grid, dim3(rgn::THREADS), 0, stream, regions, (const int*)chunk_roots, g);
    UAPS_LAUNCH(rgn::regions_relabel_kernel, chunk_grid, dim3(rgn::THREADS), 0, stream, labels, uncertainty, regions, stats,
                unc_sums, max_regions, g);
    if (unc_sums != nullptr) {
        const long long rows = (long long)B * max_regions;
        UAPS_LAUNCH(rgn::regions_means_kernel, dim3((unsigned)ceil_div<long long>(rows, rgn::THREADS)), dim3(rgn::THREADS), 0,
                    stream, (const int*)count, stats, (const double*)unc_sums, B, max_regions);
    }
    return UAPS_OK;
}
