// ants_reset.cuh -- sm_100a device code of ants_generate_env_maps: a new episode's map written straight into the cell
// records (EnvironmentGenerator.generate, environment_generator.py:60-72, with CirclesGenerator maps).
//
// One CTA per (env, tile of 64 x 64 cells = 8 x 8 record blocks).  The host hands over the random draws only: the
// anthill disc and, per env, the wall and food discs (xc, yc, r).  A CTA
//   1. culls the env's discs to those whose bounding box meets the tile (an exact integer test; a union does not care
//      about order) and compacts the survivors into shared memory, one chunk of discs at a time;
//   2. tests each of its cells against the short list:  wall = some wall disc covers the cell and the anthill disc
//      does not (walls[area] = False), food = 1 where some food disc covers a cell that is not a wall;
//   3. writes every record of the tile exactly once with 16-byte stores, nothing read from the old map: pheromone 0,
//      explored 0, occupancy 0, the wall, anthill and food fields (the layouts of st_wall / st_hill / st_food /
//      st_explored / st_occ / phero_store in ants_kernels.cuh), all timestamps 0.
// Empty pheromone fields and a 0 explored / occupancy stamp read the same under any lazy or generation counter, so the
// host counters keep running.  8-byte records keep stale side-array slots: no code of the new map escapes to them.
// With diffusion the current pheromone planes are zeroed too, with the wall bit in the sign (what k_plane_walls does).
//
// A layer may instead be Perlin noise (PerlinGenerator, the reference's default walls): the instantiation with PERLIN set
// computes the noise of the tile's cells (ants_perlin.cuh, the function ants_perlin_noise uses too) and sets the layer's
// bit where (double)noise > density; the disc list then holds the other layer's discs only.
#pragma once

#include "ants_perlin.cuh"

namespace ants {

constexpr int kResetTile = 64;                 // cells per tile side (8 record blocks)
constexpr int kResetThreads = 256;
constexpr int kResetChunk = 1024;              // discs culled per pass (the shared list holds at most one chunk)
constexpr int kResetPairs = kResetTile * kResetTile / 2 / kResetThreads;   // record pairs per thread
static_assert(kPerlinTile == kResetTile && kPerlinThreads == kResetThreads, "perlin_tile covers the reset tile");

struct ResetArgs {
    const int4 *discs;      // [n_env][kw + kf] (xc, yc, r, 0): the wall discs of an env, then its food discs
    int32_t kw, kf;         // discs per env
    int32_t env0;           // first env of the window
    int32_t tiles_x, tiles_y;
};

struct ResetPerlin {        // Perlin layers of k_reset_maps<RB, true> (offsets NULL: the layer is discs)
    PerlinArgs wall, food;
};

// sets bit k of `bits` where value k of the tile's noise exceeds the layer's density
template <int PAIRS>
__device__ __forceinline__ void perlin_layer_bits(PerlinSmem &s, const PerlinArgs &L, int el, int x0, int y0, int W,
                                                  int H, uint32_t &bits) {
    float v[2 * PAIRS];
    perlin_tile<PAIRS>(s, L, el, x0, y0, W, H, v);
#pragma unroll
    for (int k = 0; k < 2 * PAIRS; ++k)
        if ((double)v[k] > L.density) bits |= 1u << k;
}

// 64-bit word i of a record with the given fields (food 0 or 1); RB = record bytes
template <int RB>
__device__ __forceinline__ unsigned long long reset_word(const Params &p, int i, bool wall, bool hill, bool food) {
    if (RB == 8)    // {u16 ph0, u16 ph1, u16 food, u8 hill << 7 | occ, u8 wall << 7 | explored}
        return ((unsigned long long)((food ? 1u : 0u) | (hill ? 0x800000u : 0u) | (wall ? 0x80000000u : 0u))) << 32;
    if (RB == 16) { // {f32 ph0, f32 ph1, f32 food, u8 hill << 7 | occ, u8 wall << 7 | explored, u8 ts0, u8 ts1}
        if (i == 0) return 0ull;
        return (unsigned long long)(food ? 0x3F800000u : 0u) |
               ((unsigned long long)((hill ? 0x80u : 0u) | (wall ? 0x8000u : 0u)) << 32);
    }
    // f64: {f64 phero[P]; f64 food; u32 meta; u8 wall | hill << 1; timestamps}
    unsigned long long w = 0ull;
    if (i == (p.food_off >> 3) && food) w = 0x3FF0000000000000ull;
    if (i == (p.wall_off >> 3)) w |= (unsigned long long)((wall ? 1u : 0u) | (hill ? 2u : 0u)) << ((p.wall_off & 7) * 8);
    return w;
}

template <int RB, bool PERLIN = false>
__global__ void __launch_bounds__(kResetThreads) k_reset_maps(Params p, ResetArgs a, ResetPerlin pl) {
    __shared__ int4 list[kResetChunk];
    __shared__ int n_list;
    const int tiles = a.tiles_x * a.tiles_y;
    const int el = blockIdx.x / tiles, t = blockIdx.x - el * tiles;
    const int e = a.env0 + el;
    const int tx = t / a.tiles_y, ty = t - tx * a.tiles_y;
    const int x0 = tx * kResetTile, y0 = ty * kResetTile;
    const int32_t *hl = p.hill + 4 * e;
    const int4 *discs = a.discs + (int64_t)el * (a.kw + a.kf);

    // the thread's cells: record pairs j = i * threads + tid of the tile, in memory order (8 block columns of 8 blocks)
    uint32_t wall_bits = 0u, food_bits = 0u;
    const int nd = a.kw + a.kf;
    for (int c0 = 0; c0 < nd; c0 += kResetChunk) {
        if (threadIdx.x == 0) n_list = 0;
        __syncthreads();
        int4 v[kResetChunk / kResetThreads];           // (all loads of the chunk in flight before the first test)
#pragma unroll
        for (int u = 0; u < kResetChunk / kResetThreads; ++u) {
            const int d = c0 + u * kResetThreads + (int)threadIdx.x;
            v[u] = d < nd ? discs[d] : make_int4(0, 0, -1, 0);
        }
#pragma unroll
        for (int u = 0; u < kResetChunk / kResetThreads; ++u) {
            const int d = c0 + u * kResetThreads + (int)threadIdx.x;
            if (v[u].z >= 0 && v[u].x + v[u].z >= x0 && v[u].x - v[u].z < x0 + kResetTile && v[u].y + v[u].z >= y0 &&
                v[u].y - v[u].z < y0 + kResetTile) {
                v[u].w = d < a.kw ? 1 : 0;
                list[atomicAdd(&n_list, 1)] = v[u];
            }
        }
        __syncthreads();
        const int n = n_list;
        for (int s = 0; s < n; ++s) {
            const int4 c = list[s];
            const int r2 = c.z * c.z;
#pragma unroll
            for (int i = 0; i < kResetPairs; ++i) {
                const int q = 2 * (i * kResetThreads + (int)threadIdx.x);
                const int x = x0 + ((q >> 9) << 3) + ((q >> 3) & 7), y = y0 + (((q >> 6) & 7) << 3) + (q & 7);
                const int dx = c.x - x, dy0 = c.y - y, dy1 = dy0 - 1;
                const uint32_t hit = (dx * dx + dy0 * dy0 <= r2 ? 1u : 0u) | (dx * dx + dy1 * dy1 <= r2 ? 2u : 0u);
                if (c.w) wall_bits |= hit << (2 * i); else food_bits |= hit << (2 * i);
            }
        }
        __syncthreads();
    }
    if constexpr (PERLIN) {
        __shared__ PerlinSmem ps;
        if (pl.wall.offsets) perlin_layer_bits<kResetPairs>(ps, pl.wall, el, x0, y0, p.W, p.H, wall_bits);
        if (pl.food.offsets) perlin_layer_bits<kResetPairs>(ps, pl.food, el, x0, y0, p.W, p.H, food_bits);
    }

    const int nbx = p.Wp >> 3;
    uint8_t *const env_cells = p.cells + (((int64_t)e * p.plane) << p.rec_shift);
#pragma unroll
    for (int i = 0; i < kResetPairs; ++i) {
        const int q = 2 * (i * kResetThreads + (int)threadIdx.x);
        const int bx = (x0 >> 3) + (q >> 9), by = (y0 >> 3) + ((q >> 6) & 7);
        if (bx >= nbx || by >= p.nby) continue;
        const int x = (bx << 3) + ((q >> 3) & 7), y = (by << 3) + (q & 7);
        const bool in_map0 = x < p.W && y < p.H, in_map1 = x < p.W && y + 1 < p.H;
        const bool h0 = in_map0 && in_hill(hl, x, y), h1 = in_map1 && in_hill(hl, x, y + 1);
        const bool w0 = in_map0 && !h0 && ((wall_bits >> (2 * i)) & 1u), w1 = in_map1 && !h1 && ((wall_bits >> (2 * i)) & 2u);
        const bool f0 = in_map0 && !w0 && ((food_bits >> (2 * i)) & 1u), f1 = in_map1 && !w1 && ((food_bits >> (2 * i)) & 2u);
        const int cell = ((bx * p.nby + by) << 6) | (q & 63);
        uint4 *dst = reinterpret_cast<uint4 *>(env_cells + ((int64_t)cell << p.rec_shift));
        if (RB == 8) {
            const unsigned long long r0 = reset_word<8>(p, 0, w0, h0, f0), r1 = reset_word<8>(p, 0, w1, h1, f1);
            dst[0] = make_uint4((uint32_t)r0, (uint32_t)(r0 >> 32), (uint32_t)r1, (uint32_t)(r1 >> 32));
        } else {
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                const bool wl = c ? w1 : w0, hi = c ? h1 : h0, fd = c ? f1 : f0;
#pragma unroll
                for (int k = 0; k < RB / 16; ++k) {
                    const unsigned long long lo = reset_word<RB>(p, 2 * k, wl, hi, fd), hw = reset_word<RB>(p, 2 * k + 1, wl, hi, fd);
                    dst[c * (RB / 16) + k] = make_uint4((uint32_t)lo, (uint32_t)(lo >> 32), (uint32_t)hw, (uint32_t)(hw >> 32));
                }
            }
        }
        if (p.diffuse) {                               // the planes: value 0, sign = wall bit (k_plane_walls)
            for (int k = 0; k < p.P; ++k)
                *reinterpret_cast<double2 *>(plane_at(p, e, k, x, y)) = make_double2(w0 ? -0.0 : 0.0, w1 ? -0.0 : 0.0);
        }
    }
}

}  // namespace ants
