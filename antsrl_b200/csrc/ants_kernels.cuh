// ants_kernels.cuh -- sm_100a device code of the AntsRL step loop (one batch of E independent environments).
//
// Design (see DESIGN.md).  Ant-centric flat kernels over all E*N ants; the map of every environment is ONE array
// of cell records (array of structures) stored in 8 x 8-cell blocks, in one of two formats:
//     F64      (P <= 2: 32 B = one DRAM sector, P <= 4: 64 B)  { f64 phero[P]; f64 food; u32 meta; u8 wall|hill<<1; ts }
//              meta = (occ_gen << 16) | explored_gen
//     COMPACT  16 B = half a sector, the whole cell in one 128-bit load (lazy field, P <= 2)
//              { f32 phero0; f32 phero1; f32 food; u8 hill<<7|occ_gen; u8 wall<<7|explored_gen; u8 ts0; u8 ts1 }
// so a perception sample costs one load instead of five scattered plane reads.  (With DIFFUSE_FACTOR != 0 the
// pheromone field lives in two row-major f64 planes instead, for the TMA-tiled stencil: k_diffuse_tma.)
// The reference's "last writer wins" fancy-index scatters (quirk Q1: ants.py:116, pheromone.py:39,
// RL_api.py:141) and its gather-before-scatter exploration reward (Q7: reward_custom.py:89-93) are resolved
// without per-environment barriers through generation stamps:
//   owner[e][x][y] : u32 = (phase << 16) | ant   written with atomicMax -> the highest ant index of the current
//                    scatter phase owns the cell (food pickup/drop, pheromone deposit)
//   occ_gen == current step                       => an ant stands on the cell ("ants" perception channel)
//   explored_gen == 0 or == this observation      => the cell was unexplored before this observation
// The dominant kernel for the generator's channel lists is in ants_perceive_rows.cuh; k_perceive below is the
// general one (any perceived_objects list, any radius, tiny maps).
// All position / angle / sample-coordinate arithmetic is f64 in the reference's operation order (compiled with
// -fmad=false) so that truncated / rounded cell indices agree with numpy.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace ants {

constexpr int kMaxCh = 16;
constexpr int kTile = 16;                 // pheromone activity tile: 16 x 16 cells
constexpr int kGridShift = 4;             // rock grid cell = 16 x 16 map cells

struct Params {
    int32_t E, N, W, H, Hp, P, R;
    int32_t Wp, nby;                       // padded width (multiple of 8), 8x8 blocks per map row of blocks (Hp / 8)
    int64_t EN;                            // E * N
    int64_t plane;                         // Wp * Hp cells per env
    int32_t radius, S, S2, C;
    int32_t has_mask;
    int32_t ch_kind[kMaxCh];
    int32_t ch_arg[kMaxCh];
    int32_t rule_n;
    int32_t rule_op[kMaxCh];               // mandible rule in perceived_objects order: 0 = food OR, 1 = anthill AND
    int32_t reward_kind, explore_on, has_max_val;
    int32_t tiles_x, tiles_y;              // activity tiles per env
    int32_t rec_shift;                     // log2(record bytes): 4 (compact), 5 or 6
    int32_t rec16;                         // 1 = compact 16-byte record {f32 ph0, f32 ph1, f32 food, u8 occ, u8 wall|explored, u8 ts0, u8 ts1}
    int32_t rec8;                          // 1 = compact 8-byte record {u16 ph0, u16 ph1, u16 food, u8 hill|occ, u8 wall|explored}
    float *side_val;                       // rec8: [cells][3] f32 values of escaped fields (plain pheromones, non-integer food)
    uint8_t *side_ts;                      // rec8: [cells][2] write timestamps of plain pheromone values
    uint32_t ts_mask, explored_old;        // timestamp range (0xFFF / 0xFF); "explored long ago" stamp (0xFFFF / 0x7F)
    int32_t food_off, meta_off, wall_off;  // byte offsets inside a record (phero k at 8k)
    int32_t grid_w, grid_h;                // rock grid dims
    double delta, fwd_delta, reward_threshold, max_speed, max_rot_speed, csr, bsr;
    double f_explore, f_food, f_anthill, f_explore_hold, f_heading;
    double filt_center, filt_ring, phero_max_val, max_hold;
    double log2_keep;                      // log2(filt_center): lazy decay of values that are not on the table
    int32_t lazy;                          // 1 = pheromone values carry write timestamps, no evaporation pass
    int32_t ts_off;                        // P > 2: byte offset of the u16 timestamps (P <= 2: packed next to the wall byte)
    const double *decay_table;             // [tab_len] max_val decayed k times exactly like the reference
    const float *decay_obs;                // [tab_len] (float)(decay_table[k] / max_val): what the f32 observation shows
    int32_t tab_len;                       // entries until the table reaches 0 (capped)
    uint64_t rng_seed;
    int64_t env_id_base;
    // ants, [E*N]
    double *x, *y, *theta, *prev_x, *prev_y, *prev_theta, *holding, *seed;
    double *act;                           // [P][E*N]
    uint8_t *mandibles, *reward_state;
    double *rw_holding_prev, *rw_prev_dist, *rewards;
    // map
    uint8_t *cells;                        // [E][W][Hp] records
    uint32_t *owner;                       // [E][W][Hp]
    // DIFFUSE_FACTOR != 0: the pheromone field lives in two row-major f64 planes [E][P][Wp][Hp] (ping-pong: the 3x3
    // stencil reads `phero_pl` through TMA and writes `phero_alt`, then the host swaps them); the sign bit of a plane
    // value is the cell's wall bit (walls.py:30 zeroes the stencil's inputs in wall cells), its magnitude the value
    double *phero_pl, *phero_alt;
    int32_t diffuse;
    uint8_t *tile_active;                  // [E][tiles_x][tiles_y]
    int32_t *hill;                         // [E][4] = x, y, r, r*r
    double *hill_food;                     // [E]
    double *rock_c, *rock_rad, *rock_w;    // [E][R][2], [E][R], [E][R]
    unsigned long long *rock_grid;         // [E][grid_w][grid_h] bitmask of rocks near each 16x16 block
    uint32_t *rock_touch;                  // [E][R] bit c: an ant of ant-chunk c touches the rock this update
    const double *samp_off;                // [S] = (k - r) * DELTA  (RL_api.py:92-93)
    const uint8_t *mask;                   // [S2]
    double off_c[16];                      // the same offsets in the kernel-parameter constant bank
    uint32_t mask_rows[16];                // bit j of entry i = mask[i][j] (all ones without a mask)
    // scratch
    double *food_delta;                    // [E*N]
    uint32_t *commit_list, *commit_count;  // ants whose mandible action changes the food of a cell this step;
                                           // commit_count[2]: a step appends under one counter, k_food_commit zeroes the other
    uint32_t *absorb_list, *absorb_count;  // (env, cell) pairs of food lying inside the anthill disc; absorb_count[2]:
                                           // the step appends under one counter while the update zeroes the other
    uint8_t *wall_hit;                     // [E*N] 1 = the ant stands in a wall cell after this step's move
    unsigned long long *tile_counter;      // tiles processed by the evaporation kernel
    uint32_t *plain_flag;                  // lazy mode: set once any plain (non-saturated) pheromone value is stored
};

// ------------------------------------------------------------------------------------------------ helpers
__device__ __forceinline__ double pymod(double a, double b) {      // np.mod on floats (npy_remainder)
    double r = fmod(a, b);
    if (r != 0.0) {
        if ((b < 0.0) != (r < 0.0)) r += b;
    } else {
        r = copysign(0.0, b);
    }
    return r;
}
// the same value for any a; straight-line for -b < a < 2b (b > 0), which is every call of the step loop: positions
// move by at most a few cells per step and headings by less than a turn.  fmod is exact, so a - b (Sterbenz) and the
// single rounding of a + b are what npy_remainder produces.
__device__ __forceinline__ double pymod_near(double a, double b) {
    if (a >= 0.0 && a < b) return a + 0.0;              // (-0.0 -> +0.0 like copysign(0, b))
    if (a >= b && a < b + b) return a - b;
    if (a < 0.0 && a > -b) return a + b;
    return pymod(a, b);
}
__device__ __forceinline__ int imod(int a, int n) {                // np.mod on ints
    int r = a % n;
    return r < 0 ? r + n : r;
}
// ndarray.astype(int) of a coordinate in [0, n]; n itself (quirk Q14: np.mod can return exactly n) maps to
// cell 0, as the reference's own occupancy map does (RL_api.py:137-139).
__device__ __forceinline__ int cell_of(double v, int n) {
    int c = (int)v;
    return c >= n ? c - n : c;
}
__device__ __forceinline__ bool in_hill(const int32_t *hl, int cx, int cy) {   // anthill.py:31-33 on integers
    int dx = hl[0] - cx, dy = hl[1] - cy;
    return dx * dx + dy * dy <= hl[3];
}
// wrap an integer sample coordinate onto the torus (np.mod on ints); the fast path covers |offset| < n
__device__ __forceinline__ int wrap_coord(int v, int n) {
    if (v < 0) v += n; else if (v >= n) v -= n;
    return ((unsigned)v < (unsigned)n) ? v : imod(v, n);
}
// Cells are stored in 8 x 8 blocks (64 records = 2 KB contiguous, for DRAM row locality of the 7x7 perception
// windows): index of cell (x, y) inside its environment.
__device__ __forceinline__ int cidx(const Params &p, int x, int y) {
    return ((((x >> 3) * p.nby) + (y >> 3)) << 6) | ((x & 7) << 3) | (y & 7);
}
// cell record accessors
__device__ __forceinline__ uint8_t *rec_at(const Params &p, int e, int cell) {
    return p.cells + (((int64_t)e * p.plane + cell) << p.rec_shift);
}
// (f64 records only: the eager evaporation / stencil kernels)
__device__ __forceinline__ double *rec_phero(uint8_t *r, int k) { return reinterpret_cast<double *>(r) + k; }
__device__ __forceinline__ uint8_t *rec_wall(const Params &p, uint8_t *r) { return r + p.wall_off; }
// field access for both record formats.  Compact record (lazy mode, P <= 2), 16 bytes = half a sector:
//   [0] f32 phero0  [4] f32 phero1  [8] f32 food  [12] u8 (hill << 7 | occ_gen)  [13] u8 (wall << 7 | explored_gen)
//   [14],[15] u8 ts.  "hill" = the cell lies in the anthill disc (anthill.py:31-33), written by k_hill_mark at import;
//   f64 records keep it in bit 1 of the wall byte.
// Compact 8-byte record (lazy mode, P <= 2), four cells per DRAM sector:
//   [0] u16 phero0  [2] u16 phero1  [4] u16 food  [6] u8 (hill << 7 | occ_gen)  [7] u8 (wall << 7 | explored_gen)
//   pheromone code: 0 = nothing, 0x8000 | t = boxed saturated deposit of update t (mod 2^15), 1 = a plain value kept in
//   side_val / side_ts;  food code: 0 .. 0xFFFE = that many units (what the reference's maps hold), 0xFFFF = a
//   non-integer amount kept in side_val.  The side arrays are only touched for such escaped fields.
constexpr uint32_t kBox8 = 0x8000u, kBox8Mask = 0x7FFFu, kFoodEsc = 0xFFFFu;
__device__ __forceinline__ size_t rec8_index(const Params &p, const uint8_t *r) { return (size_t)(r - p.cells) >> 3; }
__device__ __forceinline__ double ld_food(const Params &p, const uint8_t *r) {
    if (p.rec8) {
        const uint32_t c = *reinterpret_cast<const uint16_t *>(r + 4);
        return c != kFoodEsc ? (double)c : (double)p.side_val[rec8_index(p, r) * 3 + 2];
    }
    return p.rec16 ? (double)*reinterpret_cast<const float *>(r + 8) : *reinterpret_cast<const double *>(r + p.food_off);
}
__device__ __forceinline__ void st_food(const Params &p, uint8_t *r, double v) {
    if (p.rec8) {
        if (v >= 0.0 && v < 65535.0 && v == floor(v)) {
            *reinterpret_cast<uint16_t *>(r + 4) = (uint16_t)(int)v;
        } else {
            *reinterpret_cast<uint16_t *>(r + 4) = (uint16_t)kFoodEsc;
            p.side_val[rec8_index(p, r) * 3 + 2] = (float)v;
            if (*p.plain_flag == 0u) *p.plain_flag = 1u;
        }
        return;
    }
    if (p.rec16) *reinterpret_cast<float *>(r + 8) = (float)v; else *reinterpret_cast<double *>(r + p.food_off) = v;
}
__device__ __forceinline__ double ld_phero(const Params &p, const uint8_t *r, int k) {
    return p.rec16 ? (double)reinterpret_cast<const float *>(r)[k] : reinterpret_cast<const double *>(r)[k];
}
__device__ __forceinline__ void st_phero(const Params &p, uint8_t *r, int k, double v) {
    if (p.rec16) reinterpret_cast<float *>(r)[k] = (float)v; else reinterpret_cast<double *>(r)[k] = v;
}
__device__ __forceinline__ bool ld_wall(const Params &p, const uint8_t *r) {
    if (p.rec8) return (r[7] >> 7) != 0;
    return p.rec16 ? (r[13] >> 7) != 0 : (r[p.wall_off] & 1) != 0;
}
__device__ __forceinline__ void st_wall(const Params &p, uint8_t *r, bool w) {
    if (p.rec8) { r[7] = (uint8_t)((r[7] & 0x7F) | (w ? 0x80 : 0)); return; }
    if (p.rec16) r[13] = (uint8_t)((r[13] & 0x7F) | (w ? 0x80 : 0)); else r[p.wall_off] = (uint8_t)((r[p.wall_off] & 2) | (w ? 1 : 0));
}
__device__ __forceinline__ void st_occ(const Params &p, uint8_t *r, uint32_t gen) {
    if (p.rec8) { r[6] = (uint8_t)((r[6] & 0x80u) | (gen & 0x7Fu)); return; }
    if (p.rec16) r[12] = (uint8_t)((r[12] & 0x80u) | (gen & 0x7Fu)); else reinterpret_cast<uint16_t *>(r + p.meta_off)[1] = (uint16_t)gen;
}
__device__ __forceinline__ uint32_t ld_occ(const Params &p, const uint8_t *r) {
    if (p.rec8) return r[6] & 0x7Fu;
    return p.rec16 ? (r[12] & 0x7Fu) : reinterpret_cast<const uint16_t *>(r + p.meta_off)[1];
}
__device__ __forceinline__ void st_hill(const Params &p, uint8_t *r, bool h) {
    if (p.rec8) { r[6] = (uint8_t)((r[6] & 0x7Fu) | (h ? 0x80u : 0u)); return; }
    if (p.rec16) r[12] = (uint8_t)((r[12] & 0x7Fu) | (h ? 0x80u : 0u)); else r[p.wall_off] = (uint8_t)((r[p.wall_off] & 1) | (h ? 2 : 0));
}
__device__ __forceinline__ uint32_t ld_explored(const Params &p, const uint8_t *r) {
    if (p.rec8) return r[7] & 0x7Fu;
    return p.rec16 ? (r[13] & 0x7Fu) : reinterpret_cast<const uint16_t *>(r + p.meta_off)[0];
}
__device__ __forceinline__ void st_explored(const Params &p, uint8_t *r, uint32_t gen) {
    if (p.rec8) { r[7] = (uint8_t)((r[7] & 0x80) | (gen & 0x7F)); return; }
    if (p.rec16) r[13] = (uint8_t)((r[13] & 0x80) | (gen & 0x7F)); else reinterpret_cast<uint16_t *>(r + p.meta_off)[0] = (uint16_t)gen;
}

// ---- lazy pheromone decay (DIFFUSE_FACTOR == 0): no pass over the field, values are decoded when read.
// A stored pheromone field is one of
//   0                      nothing
//   boxed(t)               quiet NaN whose 22-bit payload is the absolute update index t at which a SATURATED
//                          deposit (value == max_val: the reference's 256 > 255 case) was written.  Its value
//                          after update `now_abs` is decay_table[now_abs - t], the table holding max_val decayed
//                          k times with the reference's own rounding and < 0.01 cut (pheromone.py:44-45) -- bit
//                          exact for the whole episode, never folded.
//   plain value v          any other value, with a small write timestamp ts (8 or 12 bits); decays as
//                          v * 2^(k log2 c), k = now - ts (~1e-13 relative from the repeated product); the host
//                          folds plain values before the small counter wraps.
// Inside walls everything reads 0 one update after it was written (walls.py:30).
constexpr uint32_t kBoxMask = 0x3FFFFFu;   // 22-bit absolute step
__device__ __forceinline__ bool is_boxed32(uint32_t b) { return (b & 0xFFC00000u) == 0x7FC00000u; }
__device__ __forceinline__ uint32_t box32(uint32_t t) { return 0x7FC00000u | (t & kBoxMask); }
__device__ __forceinline__ bool is_boxed64(unsigned long long b) { return (b >> 32 & 0xFFF80000u) == 0x7FF80000u; }
__device__ __forceinline__ unsigned long long box64(uint32_t t) { return 0x7FF8000000000000ull | (t & kBoxMask); }

__device__ __forceinline__ uint32_t rec_ts(const Params &p, const uint8_t *r, int k) {
    if (p.rec8) return p.side_ts[rec8_index(p, r) * 2 + k];
    if (p.rec16) return r[14 + k];
    if (p.P <= 2) {
        uint32_t w = *reinterpret_cast<const uint32_t *>(r + p.wall_off);      // [wall u8][ts0 12b][ts1 12b]
        return (w >> (8 + 12 * k)) & 0xFFFu;
    }
    return *reinterpret_cast<const uint16_t *>(r + p.ts_off + 2 * k);
}
__device__ __forceinline__ void rec_set_ts(const Params &p, uint8_t *r, int k, uint32_t ts) {
    if (p.rec8) { p.side_ts[rec8_index(p, r) * 2 + k] = (uint8_t)ts; return; }
    if (p.rec16) { r[14 + k] = (uint8_t)ts; return; }
    if (p.P <= 2) {
        uint32_t *w = reinterpret_cast<uint32_t *>(r + p.wall_off);
        *w = (*w & ~(0xFFFu << (8 + 12 * k))) | ((ts & 0xFFFu) << (8 + 12 * k));
    } else {
        *reinterpret_cast<uint16_t *>(r + p.ts_off + 2 * k) = (uint16_t)(ts & 0xFFFu);
    }
}
// value of a saturated deposit of age `age` updates
__device__ __forceinline__ double boxed_value(const Params &p, uint32_t age, bool wall) {
    if (wall && age) return 0.0;
    return age < (uint32_t)p.tab_len ? p.decay_table[age] : 0.0;
}
// value of a plain stored number
__device__ __forceinline__ double plain_value(const Params &p, double v, uint32_t ts, uint32_t now, bool wall) {
    if (v == 0.0) return 0.0;
    const uint32_t k = (now - ts) & p.ts_mask;
    if (k == 0u) return v;
    if (wall) return 0.0;
    const double r = v * exp2((double)k * p.log2_keep);
    return r < 0.01 ? 0.0 : r;
}
// current value of pheromone k of record r (any format; eager modes store plain numbers without decay)
__device__ __forceinline__ double phero_value(const Params &p, const uint8_t *r, int k, uint32_t now, uint32_t now_abs) {
    if (p.rec8) {
        const uint32_t c = reinterpret_cast<const uint16_t *>(r)[k];
        if (c == 0u) return 0.0;
        const bool wl = (r[7] >> 7) != 0;
        if (c & kBox8) return boxed_value(p, (now_abs - c) & kBox8Mask, wl);
        const size_t ri = rec8_index(p, r);
        return plain_value(p, (double)p.side_val[ri * 3 + k], p.side_ts[ri * 2 + k], now, wl);
    }
    if (p.rec16) {
        const uint32_t b = reinterpret_cast<const uint32_t *>(r)[k];
        if (b == 0u) return 0.0;
        const bool wl = (r[13] >> 7) != 0;
        if (is_boxed32(b)) return boxed_value(p, (now_abs - b) & kBoxMask, wl);
        return plain_value(p, (double)__uint_as_float(b), r[14 + k], now, wl);
    }
    const unsigned long long b = reinterpret_cast<const unsigned long long *>(r)[k];
    if (!p.lazy) return __longlong_as_double((long long)b);
    if (b == 0ull) return 0.0;
    const bool wl = (r[p.wall_off] & 1) != 0;
    if (is_boxed64(b)) return boxed_value(p, (now_abs - (uint32_t)b) & kBoxMask, wl);
    return plain_value(p, __longlong_as_double((long long)b), rec_ts(p, r, k), now, wl);
}
// store a pheromone value that is current at (now, now_abs)
__device__ __forceinline__ void phero_store(const Params &p, uint8_t *r, int k, double v, uint32_t now, uint32_t now_abs) {
    if (p.rec8) {
        uint16_t *c = reinterpret_cast<uint16_t *>(r) + k;
        if (p.has_max_val && v == p.phero_max_val) { *c = (uint16_t)(kBox8 | (now_abs & kBox8Mask)); return; }
        if (v == 0.0) { *c = 0; return; }
        const size_t ri = rec8_index(p, r);
        *c = 1;
        p.side_val[ri * 3 + k] = (float)v;
        p.side_ts[ri * 2 + k] = (uint8_t)now;
        if (*p.plain_flag == 0u) *p.plain_flag = 1u;
        return;
    }
    if (p.lazy && p.has_max_val && v == p.phero_max_val) {
        if (p.rec16) reinterpret_cast<uint32_t *>(r)[k] = box32(now_abs);
        else reinterpret_cast<unsigned long long *>(r)[k] = box64(now_abs);
        return;
    }
    if (p.rec16) reinterpret_cast<float *>(r)[k] = (float)v; else reinterpret_cast<double *>(r)[k] = v;
    if (p.lazy) {
        rec_set_ts(p, r, k, now);
        if (v != 0.0 && *p.plain_flag == 0u) *p.plain_flag = 1u;
    }
}

// diffusion mode: plane accessors
__device__ __forceinline__ double *plane_at(const Params &p, int e, int k, int x, int y) {
    return p.phero_pl + ((int64_t)e * p.P + k) * p.plane + (int64_t)x * p.Hp + y;
}
__device__ __forceinline__ double plane_value(const Params &p, int e, int k, int x, int y) { return fabs(*plane_at(p, e, k, x, y)); }

// Philox4x32-10, counter (ant, step, env, 0), key (seed_lo, seed_hi) -> one double in [0,1) built like
// numpy's random_sample: ((a >> 5) * 2^26 + (b >> 6)) / 2^53.  Mirrored by oracle.philox_uniform.
__device__ __forceinline__ double philox_uniform(uint64_t seed, uint32_t env, uint32_t step, uint32_t ant) {
    uint32_t c0 = ant, c1 = step, c2 = env, c3 = 0u;
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    double a = (double)(c0 >> 5), b = (double)(c1 >> 6);
    return (a * 67108864.0 + b) / 9007199254740992.0;
}

// Programmatic dependent launch (the step kernels are launched with programmatic stream serialisation): a kernel lets
// the next one in the stream be scheduled while its own last blocks still run, and waits for its predecessor's memory
// before it touches anything.  Both are no-ops in a plain launch.
__device__ __forceinline__ void pdl_begin() {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
}

// The exploration branch of the reference's agents (collect_agent.py:172-177): rotation = randint(0, n_rot) -
// n_rot // 2, pheromone = randint(0, n_ph), per ant, drawn on the device so that neither observations nor actions cross
// PCIe.  Philox4x32-10 with counter (ant, step, env, 1) -- word 3 separates the stream from the collision noise --
// and key (seed_lo, seed_hi); value = (r * n) >> 32.  Mirrored by oracle.philox_actions.
__global__ void __launch_bounds__(256)
k_sample_actions(Params p, uint64_t seed, uint32_t step, int n_rot, int n_ph, int8_t *__restrict__ rot, int8_t *__restrict__ ph) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.EN) return;
    const int e = (int)(i / p.N);
    uint32_t c0 = (uint32_t)(i - (int64_t)e * p.N), c1 = step, c2 = (uint32_t)(p.env_id_base + e), c3 = 1u;
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    if (rot) rot[i] = (int8_t)((int)__umulhi(c0, (uint32_t)n_rot) - n_rot / 2);
    if (ph) ph[i] = (int8_t)__umulhi(c1, (uint32_t)n_ph);
}

// shared -> global bulk copy through the async proxy (TMA 1-D bulk store, SASS UBLKCP)
__device__ __forceinline__ void bulk_store_s2g(void *gdst, const void *ssrc, uint32_t bytes) {
    // the observations are written once and never read by the step loop: evict-first keeps them from displacing
    // cell records in L2 (measured: -1 % on the perception kernel)
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;\n" ::"l"(gdst),
                 "r"((uint32_t)__cvta_generic_to_shared(ssrc)), "r"(bytes), "l"(pol)
                 : "memory");
    asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
}
template <int PENDING = 0>
__device__ __forceinline__ void bulk_store_wait_read() {   // until at most PENDING bulk stores still read shared memory
    asm volatile("cp.async.bulk.wait_group.read %0;\n" ::"n"(PENDING) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
}

// Candidate rocks of a point: every rock whose (radius + reach) box overlaps the point's grid cell was OR-ed
// into that cell by rock_grid_mark, so one 8-byte load replaces a loop over all rocks.
__device__ __forceinline__ unsigned long long rock_candidates(const Params &p, int e, double x, double y) {
    int gx = cell_of(pymod_near(x, (double)p.W), p.W) >> kGridShift;
    int gy = cell_of(pymod_near(y, (double)p.H), p.H) >> kGridShift;
    return p.rock_grid[((int64_t)e * p.grid_w + gx) * p.grid_h + gy];
}
// reach of a rock in the grid: radius + the farthest a perception sample can lie from the (shifted) ant position
__device__ __forceinline__ double rock_reach(const Params &p, double rad) {
    return rad + ((double)p.radius * p.delta * 1.4142135623730951 + 1.75);
}
// Grid cells (16 map cells wide; the last one of an axis is narrower when the map size is not a multiple of 16) that
// the interval [lo, hi] of unwrapped coordinates overlaps on a torus of n cells.  grid_first / grid_next walk them:
//     for (int x = grid_first(lo); x <= grid_last(hi); x = grid_next(x, n)) g = grid_of(x, n);
// An interval as long as the map visits every grid cell (some twice: marking is idempotent).
__device__ __forceinline__ int grid_first(double lo) { return (int)floor(lo); }
__device__ __forceinline__ int grid_last(double hi) { return (int)floor(hi); }
__device__ __forceinline__ int grid_of(int x, int n) { return imod(x, n) >> kGridShift; }
__device__ __forceinline__ int grid_next(int x, int n) {
    const int w = imod(x, n);
    const int to_cell_end = (1 << kGridShift) - (w & ((1 << kGridShift) - 1)), to_seam = n - w;
    return x + (to_cell_end < to_seam ? to_cell_end : to_seam);
}
__device__ __forceinline__ int grid_count(double lo, double hi, int n) {
    int c = 0;
    for (int x = grid_first(lo); x <= grid_last(hi); x = grid_next(x, n)) ++c;
    return c;
}
__device__ __forceinline__ void rock_grid_touch(const Params &p, int e, int r, int gx, int gy, bool set) {
    unsigned long long *g = p.rock_grid + ((int64_t)e * p.grid_w + gx) * p.grid_h + gy;
    const unsigned long long bit = 1ull << r;
    if (set) atomicOr(g, bit); else atomicAnd(g, ~bit);
}
// every grid cell the box [c - L, c + L] overlaps (on the torus: ants and their perception windows wrap, RL_api.py:118-119,
// ants.py:69-71) gets (or loses) the rock's bit; one thread
__device__ __forceinline__ void rock_grid_mark(const Params &p, int e, int r, double cx, double cy, double rad, bool set = true) {
    const double L = rock_reach(p, rad);
    for (int x = grid_first(cx - L); x <= grid_last(cx + L); x = grid_next(x, p.W))
        for (int y = grid_first(cy - L); y <= grid_last(cy + L); y = grid_next(y, p.H))
            rock_grid_touch(p, e, r, grid_of(x, p.W), grid_of(y, p.H), set);
}
// the same by a whole warp: lane = (i, j) of the box's grid cells (up to 32 of them, else lane 0 alone)
__device__ __forceinline__ void rock_grid_mark_warp(const Params &p, int e, int r, double cx, double cy, double rad, bool set, int lane) {
    const double L = rock_reach(p, rad);
    const int nx = grid_count(cx - L, cx + L, p.W), ny = grid_count(cy - L, cy + L, p.H);
    if (nx * ny > 32) {
        if (lane == 0) rock_grid_mark(p, e, r, cx, cy, rad, set);
        return;
    }
    if (lane < nx * ny) {
        const int i = lane / ny, j = lane - i * ny;
        int x = grid_first(cx - L), y = grid_first(cy - L);
        for (int k = 0; k < i; ++k) x = grid_next(x, p.W);
        for (int k = 0; k < j; ++k) y = grid_next(y, p.H);
        rock_grid_touch(p, e, r, grid_of(x, p.W), grid_of(y, p.H), set);
    }
}

// ------------------------------------------------------------------------------------------------ step, part 1
// RLApi.step lines 178-196 for every ant: mandible rule, pickup / drop bookkeeping (ants.py:102-117),
// pheromone activation (ants.py:89-96), rotation (ants.py:62-67), forward move on the torus (ants.py:69-80),
// plus the occupancy stamp consumed by the "ants" perception channel (RL_api.py:136-142).
__global__ void __launch_bounds__(256)
k_step_move(Params p, const int8_t *__restrict__ rot, const int8_t *__restrict__ ph, uint32_t owner_stamp,
            uint32_t occ_gen, int all_stamp, double act_on, int cpar) {
    pdl_begin();
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.EN) return;
    int e = (int)(i / p.N);
    int a = (int)(i - (int64_t)e * p.N);
    double x = p.x[i], y = p.y[i], th = p.theta[i];
    double hold = p.holding[i];
    int m_old = p.mandibles[i] != 0;
    int pcx = cell_of(p.prev_x[i], p.W), pcy = cell_of(p.prev_y[i], p.H);      // RL_api.py:178
    int pcell = cidx(p, pcx, pcy);
    double f = ld_food(p, rec_at(p, e, pcell));
    const int32_t *hl = p.hill + 4 * e;
    bool hill = in_hill(hl, cell_of(x, p.W), cell_of(y, p.H));                  // RL_api.py:184
    int m = m_old;
    for (int k = 0; k < p.rule_n; ++k) {                                        // RL_api.py:180-184 (Q5)
        if (p.rule_op[k] == 0) m |= (f > 0.0) ? 1 : 0;
        else m &= hill ? 0 : 1;
    }
    bool closing = m && !m_old, opening = !m && m_old;                          // ants.py:103-104
    double taken = closing ? fmin(p.max_hold, fmax(0.0, f)) : 0.0;              // ants.py:111
    double dropped = opening ? hold : 0.0;                                      // ants.py:114
    double delta = dropped - taken;
    hold = hold + (taken - dropped);                                            // ants.py:117
    // ants.py:116 `qte[xy] += dropped - taken`: the highest ant index standing in the cell wins (Q1).  Ants in
    // a cell that holds no food and is outside the hill cannot change it and need not compete.
    if (all_stamp || f > 0.0 || hill) atomicMax(p.owner + (int64_t)e * p.plane + pcell, owner_stamp | (uint32_t)a);
    if (delta != 0.0) {
        uint32_t slot = atomicAdd(p.commit_count + cpar, 1u);
        p.commit_list[slot] = (uint32_t)i;
        p.food_delta[i] = delta;
    }
    p.mandibles[i] = (uint8_t)m;
    p.holding[i] = hold;
    if (ph != nullptr) {                                                        // ants.py:89-96
        int v = ph[i];
        p.act[i] = (v == 1) ? act_on : 0.0;
        p.act[p.EN + i] = (v != 0 && v != 1) ? act_on : 0.0;
    }
    if (rot != nullptr) th = pymod_near(th + (double)rot[i] * p.max_rot_speed, 6.283185307179586);   // ants.py:62-67
    double fwd = (1.0 * p.max_speed) * (1.0 - hold * p.csr);                    // RL_api.py:194
    if (fwd < 0.0) fwd *= p.bsr;                                                // RL_api.py:195
    double s, c;
    sincos(th, &s, &c);
    x = pymod_near(x + c * fwd, (double)p.W);                                   // ants.py:69-80
    y = pymod_near(y + s * fwd, (double)p.H);
    p.x[i] = x; p.y[i] = y; p.theta[i] = th;
    uint8_t *orec = rec_at(p, e, cidx(p, cell_of(x, p.W), cell_of(y, p.H)));
    p.wall_hit[i] = ld_wall(p, orec) ? 1 : 0;           // read here for Walls.update: k_collide then needs no record
    st_occ(p, orec, occ_gen);
}

// Occupancy stamp alone, for a stand-alone observation() (main.py:88).
__global__ void __launch_bounds__(256) k_occ_stamp(Params p, uint32_t occ_gen) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.EN) return;
    int e = (int)(i / p.N);
    uint8_t *orec = rec_at(p, e, cidx(p, cell_of(p.x[i], p.W), cell_of(p.y[i], p.H)));
    st_occ(p, orec, occ_gen);
}

// ------------------------------------------------------------------------------------------------ step, part 2
// The winners of the food scatter write `old + (dropped - taken)` (ants.py:116); food that now lies inside the
// anthill disc is queued for Anthill.update (anthill.py:41-46).
__global__ void __launch_bounds__(128) k_food_commit(Params p, uint32_t owner_stamp, int par, int cpar) {
    pdl_begin();
    uint32_t n = p.commit_count[cpar];
    if (blockIdx.x == 0 && threadIdx.x == 0) p.commit_count[cpar ^ 1] = 0u;    // for the next step
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
        int64_t i = p.commit_list[k];
        int e = (int)(i / p.N);
        int a = (int)(i - (int64_t)e * p.N);
        int pcx = cell_of(p.prev_x[i], p.W), pcy = cell_of(p.prev_y[i], p.H);
        int pcell = cidx(p, pcx, pcy);
        if (p.owner[(int64_t)e * p.plane + pcell] != (owner_stamp | (uint32_t)a)) continue;
        uint8_t *fr = rec_at(p, e, pcell);
        double nv = ld_food(p, fr) + p.food_delta[i];
        st_food(p, fr, nv);
        nv = ld_food(p, fr);                                                   // as stored (f32 in compact records)
        if (nv != 0.0 && in_hill(p.hill + 4 * e, pcx, pcy)) {
            // (the list holds E * N pairs, one step's worth: past that the update sweeps every disc instead)
            uint32_t s = atomicAdd(p.absorb_count + par, 1u);
            if (s < (uint32_t)p.EN) {
                p.absorb_list[2 * s] = (uint32_t)e;
                p.absorb_list[2 * s + 1] = (uint32_t)pcell;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------ perception + reward
// RLApi.observation (RL_api.py:96-165) fused with reward.observation (reward_custom.py) and, when called from
// step, Ants.give_reward (ants.py:119-121).
//
// LAYOUT 0: any perceived_objects list (switch per channel)
// LAYOUT 1: the generator's default list [ants, phero0, phero1, anthill, walls, food] (environment_generator.py:64-99)
// LAYOUT 2: the same plus rocks as 7th channel
//
// Block = blockDim.x threads = as many consecutive ants; warp w owns ants [32w, 32w+32) from start to end (no
// block barrier after the table load).
//   phase A (thread per ant): f64 trigonometry of the rotated sampling frame (cos/sin(theta + pi/2), shifted
//            position) into a 96-byte shared-memory record per ant; reward terms that do not need the exploration
//            count; agent_state / state outputs; candidate rocks from the rock grid.
//   phase B (warp, flat sample index): the warp walks its ants in chunks of `group` ants; the chunk's
//            group*S2 samples are spread over the 32 lanes and processed in batches of U lane-slots: sample cell =
//            round_half_even(rot * offset + xy_f) mod (W,H) in f64, then the record loads (one 32-byte sector per
//            sample) of the whole batch are issued before any is consumed; analytic anthill disc, exact rock test
//            on the candidates; exploration counts by warp-uniform ballot splitting; the chunk's
//            (group x S2 x C) f32 tile is staged in shared memory and leaves with ONE TMA bulk store.
//   phase C (thread per ant): reward epilogue and Ants.give_reward.
constexpr int kPerceiveThreads = 128;
constexpr int kMaxGroup = 4;                // ants per staged chunk (4 ants: bytes are always a multiple of 16)

struct AntPrep {                            // 96 bytes per ant, shared memory
    double ct, st;               // cos / sin(theta + pi/2)
    double xf, yf;               // position shifted forward by perception_fwd_delta
    const uint8_t *cells;        // records of the ant's environment
    unsigned long long rocks;    // candidate rocks (from the rock grid)
    int hx, hy, hr2, e;          // anthill centre, radius^2; environment index
    double r_other, mult;        // reward terms without the exploration count; exploration multiplier
};
struct SampleTab {                          // per sample of the window: offsets (RL_api.py:92-93)
    double px, py;
};

template <int LAYOUT, bool REC16>
__global__ void __launch_bounds__(kPerceiveThreads, 6)
k_perceive(Params p, float *__restrict__ obs, float *__restrict__ agent_state, float *__restrict__ state_out,
           double *__restrict__ reward_out, uint32_t obs_gen, uint32_t occ_gen, int is_step, int rw_alias,
           int group, uint32_t s2_magic, int slow_wrap, uint32_t now, uint32_t now_abs) {
    pdl_begin();
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int S = p.S, S2 = p.S2, C = p.C;
    const int SC = S2 * C;
    const int nthreads = blockDim.x, nwarps = nthreads >> 5;
    float *s_obs = reinterpret_cast<float *>(smem_raw);                        // [warps][group][S2*C], 16 B aligned
    AntPrep *prep = reinterpret_cast<AntPrep *>(s_obs + ((nwarps * group * SC + 3) & ~3));
    SampleTab *s_tab = reinterpret_cast<SampleTab *>(prep + nthreads);         // [S2]
    int *s_cnt = reinterpret_cast<int *>(s_tab + S2);
    uint8_t *s_mask = reinterpret_cast<uint8_t *>(s_cnt + nthreads);

    const int tid = threadIdx.x;
    for (int k = tid; k < S2; k += nthreads) {
        s_mask[k] = p.has_mask ? p.mask[k] : 1;
        s_tab[k].px = p.samp_off[k % S];       // X = off[j], Y = off[i] for sample k = i * S + j
        s_tab[k].py = p.samp_off[k / S];
    }
    const int64_t base = (int64_t)blockIdx.x * nthreads;

    // ---- phase A (thread per ant)
    {
        const int64_t i = base + tid;
        s_cnt[tid] = 0;
        if (i < p.EN) {
            const int e = (int)(i / p.N);
            const double x = p.x[i], y = p.y[i], th = p.theta[i], hold = p.holding[i];
            double s0, c0, st, ct;
            sincos(th, &s0, &c0);
            sincos(th + 3.141592653589793 * 0.5, &st, &ct);                    // RL_api.py:101,107-108
            AntPrep q;
            q.ct = ct; q.st = st;
            q.xf = x; q.yf = y;
            if (p.fwd_delta != 0.0) { q.xf = x + c0 * p.fwd_delta; q.yf = y + s0 * p.fwd_delta; }   // :103-104
            q.e = e;
            q.cells = p.cells + (((int64_t)e * p.plane) << p.rec_shift);
            const int32_t *hl = p.hill + 4 * e;
            q.hx = hl[0]; q.hy = hl[1]; q.hr2 = hl[3];
            // reward.observation, reward_custom.py
            const double hprev = rw_alias ? hold : p.rw_holding_prev[i];       // Q18
            const double d = hold - hprev;
            q.r_other = 0.0; q.mult = 1.0;
            if (p.reward_kind == 0) {                                          // All_Rewards, :79-106
                const double r_food = d < 0.0 ? 0.0 : d;
                const double r_hill = d < 0.0 ? 1.0 : 0.0;
                const double ddx = x - (double)q.hx, ddy = y - (double)q.hy;
                const double nd = sqrt(ddx * ddx + ddy * ddy);
                const double heading = (p.rw_prev_dist[i] > nd && hold > 0.0) ? 0.1 : 0.0;
                p.rw_prev_dist[i] = nd;
                q.r_other = r_food * p.f_food + r_hill * p.f_anthill + heading * p.f_heading;
                q.mult = (hold == 0.0) ? p.f_explore : p.f_explore_hold;
                p.rw_holding_prev[i] = hold;
            } else if (p.reward_kind == 2) {                                   // Food_Reward, :37-40
                q.r_other = d < 0.0 ? 10.0 : d;
                p.rw_holding_prev[i] = hold;
            }
            q.rocks = (p.R > 0 && (LAYOUT == 2 || LAYOUT == 0)) ? rock_candidates(p, e, q.xf, q.yf) : 0ull;
            prep[tid] = q;
            agent_state[2 * i] = (float)hold;                                  // RL_api.py:160-162
            agent_state[2 * i + 1] = (float)p.seed[i];
            if (state_out != nullptr) {                                        // RL_api.py:155-158
                float *so = state_out + i * (2 + p.P);
                so[0] = (float)p.mandibles[i];
                so[1] = (float)hold;
                for (int k = 0; k < p.P; ++k) so[2 + k] = p.act[(int64_t)k * p.EN + i] > 0.0 ? 1.f : 0.f;
            }
        }
    }
    const double inv_max = 1.0 / p.phero_max_val;   // obs is f32: x * (1/max) == x / max to well below 1e-5
    const bool has_mask = p.has_mask != 0;
    const bool explore_on = p.explore_on != 0;
    const int food_off = p.food_off, meta_off = p.meta_off, wall_off = p.wall_off, rec_shift = p.rec_shift;
    const int W = p.W, H = p.H, nby = p.nby;
    __syncthreads();

    // ---- phase B (warp, flat sample index; the warp owns ants [32 warp, 32 warp + 32) of the block)
    const int warp = tid >> 5, lane = tid & 31;
    float *wobs = s_obs + warp * group * SC;
    const AntPrep *wprep = prep + warp * 32;
    constexpr int U = 4;                       // lane-slots per batch: all record loads of a batch are in flight together
    for (int g = 0; g < 32; g += group) {
        const int64_t i0 = base + warp * 32 + g;
        if (i0 >= p.EN) break;
        int n_in = 32 - g < group ? 32 - g : group;
        if (p.EN - i0 < n_in) n_in = (int)(p.EN - i0);
        const int nsamp = n_in * S2;
        // the previous chunk's bulk store must have finished reading the staging tile
        if (lane == 0) bulk_store_wait_read();
        __syncwarp();
        const int iters = (nsamp + 31) >> 5;
        uint32_t cnt_packed = 0;               // exploration counts of the chunk's ants, one byte each (warp-uniform)
        for (int it0 = 0; it0 < iters; it0 += U) {
            uint32_t xy[U];
            const uint8_t *rp[U];
            uint4 lo[U], hi[U];                // record halves (P == 2 fast path) or generic fields packed likewise
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int f_raw = (it0 + u) * 32 + lane;
                const int f = f_raw < nsamp ? f_raw : 0;                       // idle lanes / slots shadow sample 0
                const int aj = (int)(((uint32_t)f * s2_magic) >> 20);         // f / S2
                const int s = f - aj * S2;
                const AntPrep &q = wprep[g + aj];
                const SampleTab t = s_tab[s];
                // sample cell, RL_api.py:110-119: round_half_even(rot(theta + pi/2) * offset + xy_f) mod (W, H)
                const double rx = q.ct * t.px - q.st * t.py;
                const double ry = q.st * t.px + q.ct * t.py;
                int ix = __double2int_rn(rx + q.xf), iy = __double2int_rn(ry + q.yf);
                if (slow_wrap) { ix = imod(ix, W); iy = imod(iy, H); }
                else {
                    ix = ix < 0 ? ix + W : (ix >= W ? ix - W : ix);
                    iy = iy < 0 ? iy + H : (iy >= H ? iy - H : iy);
                }
                xy[u] = ((uint32_t)ix << 16) | (uint32_t)iy;
                rp[u] = q.cells + ((int64_t)(((((ix >> 3) * nby) + (iy >> 3)) << 6) | ((ix & 7) << 3) | (iy & 7)) << rec_shift);
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (REC16) {                   // compact record: the whole cell in one 128-bit load
                    lo[u] = *reinterpret_cast<const uint4 *>(rp[u]);
                    hi[u] = make_uint4(0u, 0u, 0u, 0u);
                } else if (LAYOUT != 0) {      // P == 2: {ph0, ph1} | {food, meta, wall + timestamps}
                    lo[u] = *reinterpret_cast<const uint4 *>(rp[u]);
                    hi[u] = *reinterpret_cast<const uint4 *>(rp[u] + 16);
                } else if (p.rec8) {           // 8-byte record (this kernel serves it through LAYOUT 0 only)
                    const uint2 v8 = *reinterpret_cast<const uint2 *>(rp[u]);
                    const double fdv = (v8.y & 0xFFFFu) != kFoodEsc ? (double)(v8.y & 0xFFFFu) : ld_food(p, rp[u]);
                    const uint32_t fl = v8.y >> 16;                            // [hill|occ][wall|explored]
                    hi[u] = make_uint4((uint32_t)__double2loint(fdv), (uint32_t)__double2hiint(fdv),
                                       ((fl & 0x7Fu) << 16) | ((fl >> 8) & 0x7Fu), (fl >> 15) & 1u);
                    lo[u] = make_uint4(0u, 0u, 0u, 0u);
                } else {                       // generic f64 record: gather the fields into the same register shape
                    const double fdv = *reinterpret_cast<const double *>(rp[u] + food_off);
                    const uint32_t mtv = *reinterpret_cast<const uint32_t *>(rp[u] + meta_off);
                    const uint32_t wlv = *(rp[u] + wall_off) & 1u;
                    hi[u] = make_uint4((uint32_t)__double2loint(fdv), (uint32_t)__double2hiint(fdv), mtv, wlv);
                    lo[u] = make_uint4(0u, 0u, 0u, 0u);
                }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int f0 = (it0 + u) * 32;                                 // warp-uniform
                if (f0 >= nsamp) break;
                const int f = f0 + lane;
                const bool valid = f < nsamp;
                // fields of the record, whatever its format
                uint32_t occ, eg;
                bool wl;
                float fdf;                     // food as the f32 observation shows it
                if (REC16) {
                    const uint32_t pk = lo[u].w;
                    occ = pk & 0x7Fu; eg = (pk >> 8) & 0x7Fu; wl = ((pk >> 15) & 1u) != 0;
                    fdf = __uint_as_float(lo[u].z);
                } else {
                    occ = hi[u].z >> 16; eg = hi[u].z & 0xFFFFu; wl = (hi[u].w & 1u) != 0;
                    fdf = (float)__hiloint2double((int)hi[u].y, (int)hi[u].x);
                }
                if (explore_on) {
                    const bool unexplored = valid && ((eg == 0u) || (eg == obs_gen));     // gather-before-scatter, Q7
                    if (valid && eg == 0u) {
                        if (REC16) const_cast<uint8_t *>(rp[u])[13] = (uint8_t)((wl ? 0x80u : 0u) | obs_gen);
                        else if (p.rec8) const_cast<uint8_t *>(rp[u])[7] = (uint8_t)((wl ? 0x80u : 0u) | obs_gen);
                        else *reinterpret_cast<uint16_t *>(const_cast<uint8_t *>(rp[u]) + meta_off) = (uint16_t)obs_gen;
                    }
                    // the slot's lanes belong to consecutive ants: split the ballot at the ant boundaries (uniform)
                    uint32_t votes = __ballot_sync(0xffffffffu, unexplored);
                    int a_lo = (int)(((uint32_t)f0 * s2_magic) >> 20);
                    int covered = 0;
                    while (covered < 32) {
                        int span = (a_lo + 1) * S2 - (f0 + covered);           // lanes left in ant a_lo
                        span = span < 32 - covered ? span : 32 - covered;
                        uint32_t m = span >= 32 ? 0xffffffffu : (((1u << span) - 1u) << covered);
                        cnt_packed += (uint32_t)__popc(votes & m) << (8 * a_lo);
                        covered += span;
                        ++a_lo;
                        if (a_lo >= n_in) break;
                    }
                }
                if (!valid) continue;
                const int aj = (int)(((uint32_t)f * s2_magic) >> 20);
                const int s = f - aj * S2;
                const int ix = (int)(xy[u] >> 16), iy = (int)(xy[u] & 0xFFFFu);
                const bool vis = s_mask[s] != 0;
                float *o = wobs + f * C;
                const AntPrep &q = wprep[g + aj];
                const int hdx = q.hx - ix, hdy = q.hy - iy;
                const bool hill = hdx * hdx + hdy * hdy <= q.hr2;              // anthill.py:31-33 on integers
                // mask * (perception + 1) - 1 (RL_api.py:147-148): the +1-1 round trip changes a value by at most
                // 2^-53 absolute, far below the resolution of the f32 observation, so visible samples pass through.
                if (LAYOUT != 0) {
                    // pheromone channels, RL_api.py:124-125: zero and saturated-deposit fields (the common cases)
                    // decode without f64; anything else goes through phero_value
                    float v1, v2;
                    if (REC16) {
                        const uint32_t b0 = lo[u].x, b1 = lo[u].y;
                        if (b0 == 0u) v1 = 0.f;
                        else if (is_boxed32(b0) && !wl) { uint32_t age = (now_abs - b0) & kBoxMask; v1 = age < (uint32_t)p.tab_len ? p.decay_obs[age] : 0.f; }
                        else v1 = (float)(phero_value(p, rp[u], 0, now, now_abs) * inv_max);
                        if (b1 == 0u) v2 = 0.f;
                        else if (is_boxed32(b1) && !wl) { uint32_t age = (now_abs - b1) & kBoxMask; v2 = age < (uint32_t)p.tab_len ? p.decay_obs[age] : 0.f; }
                        else v2 = (float)(phero_value(p, rp[u], 1, now, now_abs) * inv_max);
                    } else {
                        const unsigned long long b0 = ((unsigned long long)lo[u].y << 32) | lo[u].x;
                        const unsigned long long b1 = ((unsigned long long)lo[u].w << 32) | lo[u].z;
                        if (b0 == 0ull) v1 = 0.f;
                        else if (p.lazy && is_boxed64(b0) && !wl) { uint32_t age = (now_abs - lo[u].x) & kBoxMask; v1 = age < (uint32_t)p.tab_len ? p.decay_obs[age] : 0.f; }
                        else v1 = (float)(phero_value(p, rp[u], 0, now, now_abs) * inv_max);
                        if (b1 == 0ull) v2 = 0.f;
                        else if (p.lazy && is_boxed64(b1) && !wl) { uint32_t age = (now_abs - lo[u].z) & kBoxMask; v2 = age < (uint32_t)p.tab_len ? p.decay_obs[age] : 0.f; }
                        else v2 = (float)(phero_value(p, rp[u], 1, now, now_abs) * inv_max);
                    }
                    float v0 = (occ == occ_gen) ? 1.f : 0.f;                                          // :136-142
                    float v3 = hill ? 1.f : 0.f;                                                      // :130-131
                    float v4 = wl ? 1.f : 0.f;                                                        // :128-129
                    float v5 = fdf;                                                                   // :126-127
                    float v6 = 0.f;
                    if (LAYOUT == 2) {                                                                // :132-135
                        unsigned long long rm = q.rocks;
                        if (rm) {
                            const double *rc = p.rock_c + (int64_t)q.e * p.R * 2;
                            const double *rr = p.rock_rad + (int64_t)q.e * p.R;
                            while (rm) {
                                int r = __ffsll((long long)rm) - 1;
                                rm &= rm - 1;
                                double ddx = (double)ix - rc[2 * r], ddy = (double)iy - rc[2 * r + 1];
                                if (sqrt(ddx * ddx + ddy * ddy) < rr[r]) { v6 = 1.f; break; }
                            }
                        }
                    }
                    if (!vis) { v0 = v1 = v2 = v3 = v4 = v5 = v6 = -1.f; }
                    o[0] = v0; o[1] = v1; o[2] = v2; o[3] = v3; o[4] = v4; o[5] = v5;
                    if (LAYOUT == 2) o[6] = v6;
                } else {
                    for (int c = 0; c < C; ++c) {
                        double v;
                        switch (p.ch_kind[c]) {
                            case 0: v = (occ == occ_gen) ? 1.0 : 0.0; break;
                            case 1: v = (p.diffuse ? plane_value(p, q.e, p.ch_arg[c], ix, iy)
                                                   : phero_value(p, rp[u], p.ch_arg[c], now, now_abs)) * inv_max; break;
                            case 2: v = hill ? 1.0 : 0.0; break;
                            case 3: v = wl ? 1.0 : 0.0; break;
                            case 4: v = (double)fdf; break;
                            default: {
                                v = 0.0;
                                unsigned long long rm = q.rocks;
                                const double *rc = p.rock_c + (int64_t)q.e * p.R * 2;
                                const double *rr = p.rock_rad + (int64_t)q.e * p.R;
                                while (rm) {
                                    int r = __ffsll((long long)rm) - 1;
                                    rm &= rm - 1;
                                    double ddx = (double)ix - rc[2 * r], ddy = (double)iy - rc[2 * r + 1];
                                    if (sqrt(ddx * ddx + ddy * ddy) < rr[r]) { v = 1.0; break; }
                                }
                            }
                        }
                        o[c] = (has_mask && !vis) ? -1.f : (float)v;
                    }
                }
            }
        }
        if (explore_on && lane < n_in) s_cnt[warp * 32 + g + lane] = (int)((cnt_packed >> (8 * lane)) & 0xFFu);
        // flush the staged (n_in x S2 x C) f32 tile: one TMA bulk store when 16 B granular, else plain stores
        float *dst = obs + i0 * SC;
        const uint32_t bytes = (uint32_t)(n_in * SC * 4);
        if ((bytes & 15u) == 0 && (reinterpret_cast<uintptr_t>(dst) & 15u) == 0) {
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) bulk_store_s2g(dst, wobs, bytes);
        } else {
            __syncwarp();
            for (int t = lane; t < n_in * SC; t += 32) dst[t] = wobs[t];
            __syncwarp();
        }
    }
    __syncwarp();

    // ---- phase C: reward epilogue, thread per ant (this warp's own ants)
    {
        const int64_t i = base + tid;
        if (i < p.EN) {
            const AntPrep &q = prep[tid];
            const int count = s_cnt[tid];
            double reward;
            if (p.reward_kind == 1) {
                reward = (double)count / 10.0;                                 // reward_custom.py:19
            } else if (p.reward_kind == 0) {
                reward = 0.0;
                if (explore_on) reward += ((double)count / 10.0) * q.mult;     // :89-94
                reward += q.r_other;                                           // :106
            } else {
                reward = q.r_other;
            }
            p.rewards[i] = reward;
            if (reward_out != nullptr) reward_out[i] = reward;
            if (is_step) {                                                     // ants.py:119-121 (Q16)
                int rs = p.reward_state[i];
                rs += ((reward - p.reward_threshold) > 0.0) ? 255 : 0;
                p.reward_state[i] = (uint8_t)(rs > 255 ? 255 : rs);
            }
        }
    }
    if (lane == 0) bulk_store_wait_read();   // smem must stay valid until the last bulk store has read it
}

// ------------------------------------------------------------------------------------------------ update, ants side
// Walls.update for ants (walls.py:24-28) and, when there are no rocks, the ant part of Ants.update
// (ants.py:124,130) plus the ownership stamp of the pheromone deposit (pheromone.py:39, Q1).
__global__ void __launch_bounds__(256)
k_collide(Params p, const double *__restrict__ noise, uint32_t step_id, uint32_t owner_stamp, int finish, int use_flag,
          int par) {
    pdl_begin();
    // Anthill.update (anthill.py:41-46) for the cells queued by k_food_commit: nothing else in the update reads the
    // food field, so the first blocks of this kernel absorb them; the other counter is zeroed for the next step.  (A
    // count past E * N means the list overflowed: the update then sweeps every disc, k_absorb_sweep.)
    {
        const uint32_t n = min(p.absorb_count[par], (uint32_t)p.EN);
        const uint32_t nb = gridDim.x < 32u ? gridDim.x : 32u;
        if (blockIdx.x < nb) {
            for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += nb * blockDim.x) {
                uint32_t e = p.absorb_list[2 * k], c = p.absorb_list[2 * k + 1];
                uint8_t *fr = rec_at(p, (int)e, (int)c);
                double v;                                                      // qte -= qte * area
                if (p.rec8) {          // the food code is the low half of the record's second word
                    const uint32_t c = atomicAnd(reinterpret_cast<unsigned int *>(fr + 4), 0xFFFF0000u) & 0xFFFFu;
                    v = c != kFoodEsc ? (double)c : (double)p.side_val[rec8_index(p, fr) * 3 + 2];
                } else if (p.rec16) v = (double)__uint_as_float(atomicExch(reinterpret_cast<unsigned int *>(fr + 8), 0u));
                else v = __longlong_as_double((long long)atomicExch(reinterpret_cast<unsigned long long *>(fr + p.food_off), 0ull));
                if (v != 0.0) atomicAdd(p.hill_food + e, v);
            }
        }
        if (blockIdx.x == 0 && threadIdx.x == 0) p.absorb_count[par ^ 1] = 0u;
    }
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.EN) return;
    int e = (int)(i / p.N);
    int a = (int)(i - (int64_t)e * p.N);
    double x = p.x[i], y = p.y[i], th = p.theta[i];
    const bool in_wall = use_flag ? p.wall_hit[i] != 0
                                  : ld_wall(p, rec_at(p, e, cidx(p, cell_of(x, p.W), cell_of(y, p.H))));
    if (in_wall) {
        x = p.prev_x[i]; y = p.prev_y[i];
        double u = noise ? noise[i] : philox_uniform(p.rng_seed, (uint32_t)(p.env_id_base + e), step_id, (uint32_t)a);
        th += u - 0.5;                                                         // not re-wrapped (Q3)
        p.x[i] = x; p.y[i] = y; p.theta[i] = th;
    }
    if (p.R > 0) {
        // CircleObstacles.update, first half (circle_obstacles.py:35-37): which rocks does this ant push?  The rocks
        // registered near it in the rock grid (current centres) are tested exactly; a hit sets the bit of the ant's
        // chunk in rock_touch[e][rock] for k_rocks_pushed.
        unsigned long long rm = rock_candidates(p, e, x, y);
        if (rm) {
            const double *rc = p.rock_c + (int64_t)e * p.R * 2;
            const double *rr = p.rock_rad + (int64_t)e * p.R;
            const int G = ((p.N + 31) / 32 + 31) / 32 * 32;  // ants per chunk: a multiple of 32, at most 32 chunks
            while (rm) {
                int r = __ffsll((long long)rm) - 1;
                rm &= rm - 1;
                double vx = rc[2 * r] - x, vy = rc[2 * r + 1] - y;
                if (!(sqrt(vx * vx + vy * vy) > rr[r])) atomicOr(p.rock_touch + (int64_t)e * p.R + r, 1u << (a / G));
            }
        }
    }
    if (finish) {
        p.prev_x[i] = x; p.prev_y[i] = y; p.prev_theta[i] = th;
        atomicMax(p.owner + (int64_t)e * p.plane + cidx(p, cell_of(x, p.W), cell_of(y, p.H)), owner_stamp | (uint32_t)a);
        p.reward_state[i] = (uint8_t)((double)p.reward_state[i] * 0.9);        // ants.py:130
    }
}

// CircleObstacles.update, first half (circle_obstacles.py:35-40): ants push rocks.  One warp per (env, rock); a rock
// no ant touches (rock_touch == 0, set by k_collide) costs one load.  For a touched rock the warp walks only the
// touched ant-chunks, in ant order, adding the pushes with an ordered ballot loop -- the same summation order as
// np.sum(axis=0); untouched ants contribute exact 0.  Then the rock's entries in the rock grid move with it.
__global__ void __launch_bounds__(256) k_rocks_pushed(Params p) {
    pdl_begin();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t pair = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp;
    if (pair >= (int64_t)p.E * p.R) return;
    // the rock's data is requested together with its touch word: one memory round trip instead of three for a touched
    // rock (the arrays are small and L2-resident; an untouched rock wastes 40 bytes of L2 traffic)
    const int e = (int)(pair / p.R), r = (int)(pair - (int64_t)e * p.R);
    double *rc = p.rock_c + (int64_t)e * p.R * 2;
    uint32_t tm = p.rock_touch[pair];
    const double cx = rc[2 * r], cy = rc[2 * r + 1], rad = p.rock_rad[pair], wt = p.rock_w[pair];
    if (tm == 0u) return;
    const double *xs = p.x + (int64_t)e * p.N, *ys = p.y + (int64_t)e * p.N;
    const int G = ((p.N + 31) / 32 + 31) / 32 * 32;
    double sx = 0.0, sy = 0.0;
    while (tm) {
        const int g = __ffs(tm) - 1;
        tm &= tm - 1;
        const int a_end = min((g + 1) * G, p.N);
        for (int a0 = g * G; a0 < a_end; a0 += 32) {
            int a = a0 + lane;
            double px = 0.0, py = 0.0;
            bool hit = false;
            if (a < a_end) {
                double vx = cx - xs[a], vy = cy - ys[a];
                double d = sqrt(vx * vx + vy * vy);
                if (!(d > rad)) {
                    double fac = 1.0 - rad / (d + 0.001);
                    px = vx * fac; py = vy * fac; hit = true;
                }
            }
            unsigned m = __ballot_sync(0xffffffffu, hit);
            while (m) {
                int l = __ffs(m) - 1;
                m &= m - 1;
                sx += __shfl_sync(0xffffffffu, px, l);
                sy += __shfl_sync(0xffffffffu, py, l);
            }
        }
    }
    // every lane holds the same sums
    const double nx = cx - sx / wt, ny = cy - sy / wt;
    if (lane == 0) {
        rc[2 * r] = nx;
        rc[2 * r + 1] = ny;
        p.rock_touch[pair] = 0u;
    }
    if (nx != cx || ny != cy) {                        // the grid entries follow the rock
        rock_grid_mark_warp(p, e, r, cx, cy, rad, false, lane);
        __syncwarp();                                  // orders the clears before the sets (the boxes overlap)
        rock_grid_mark_warp(p, e, r, nx, ny, rad, true, lane);
    }
}

// CircleObstacles.update, second half (circle_obstacles.py:53-58) + the ant part of Ants.update.
__global__ void __launch_bounds__(256) k_rocks_push_ants(Params p, uint32_t owner_stamp) {
    pdl_begin();
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.EN) return;
    int e = (int)(i / p.N);
    int a = (int)(i - (int64_t)e * p.N);
    double x = p.x[i], y = p.y[i];
    const double *rc = p.rock_c + (int64_t)e * p.R * 2;
    const double *rr = p.rock_rad + (int64_t)e * p.R;
    double sx = 0.0, sy = 0.0;
    // only rocks registered in the ant's grid cell can be within their radius (the grid box is wider than that);
    // candidates are visited in rock order like np.sum(axis=1)
    unsigned long long rm = rock_candidates(p, e, x, y);
    while (rm) {
        int r = __ffsll((long long)rm) - 1;
        rm &= rm - 1;
        double vx = rc[2 * r] - x, vy = rc[2 * r + 1] - y;
        double d = sqrt(vx * vx + vy * vy);
        double rad = rr[r];
        if (!(d > rad)) {
            double fac = 1.0 - rad / (d + 0.001);
            sx += vx * fac; sy += vy * fac;
        }
    }
    x = pymod_near(x + sx, (double)p.W);                                       // translate_ants -> warp_xy
    y = pymod_near(y + sy, (double)p.H);
    p.x[i] = x; p.y[i] = y;
    p.prev_x[i] = x; p.prev_y[i] = y; p.prev_theta[i] = p.theta[i];
    atomicMax(p.owner + (int64_t)e * p.plane + cidx(p, cell_of(x, p.W), cell_of(y, p.H)), owner_stamp | (uint32_t)a);
    p.reward_state[i] = (uint8_t)((double)p.reward_state[i] * 0.9);
}

// ------------------------------------------------------------------------------------------------ pheromone field
// One cell of Walls.update's field zeroing (walls.py:30), Pheromone.update reduced to its centre tap for
// DIFFUSE_FACTOR == 0 (pheromone.py:44, bit-identical to convolve2d with an all-zero ring), the threshold of
// pheromone.py:45 and the whole-plane clamp of pheromone.py:41.  Returns true if pheromone remains.
__device__ __forceinline__ bool evaporate_record(const Params &p, uint8_t *r, double c, double mx, bool clamp) {
    bool any = false;
    if (p.P == 2) {
        double2 v = *reinterpret_cast<double2 *>(r);
        if (v.x == 0.0 && v.y == 0.0) return false;
        const bool wl = (*rec_wall(p, r) & 1) != 0;
        double a = wl ? 0.0 : v.x * c, b = wl ? 0.0 : v.y * c;
        a = a < 0.01 ? 0.0 : a;
        b = b < 0.01 ? 0.0 : b;
        if (clamp) { a = fmin(a, mx); b = fmin(b, mx); }
        *reinterpret_cast<double2 *>(r) = make_double2(a, b);
        any = (a != 0.0) || (b != 0.0);
    } else {
        const bool wl = (*rec_wall(p, r) & 1) != 0;
        for (int k = 0; k < p.P; ++k) {
            double v = *rec_phero(r, k);
            if (v == 0.0) continue;
            double a = wl ? 0.0 : v * c;
            a = a < 0.01 ? 0.0 : a;
            if (clamp) a = fmin(a, mx);
            *rec_phero(r, k) = a;
            any |= a != 0.0;
        }
    }
    return any;
}

// Dense pass over every cell of every environment.
__global__ void __launch_bounds__(256) k_evaporate_dense(Params p) {
    const int64_t n = (int64_t)p.E * p.plane;
    const double c = p.filt_center, mx = p.phero_max_val;
    const bool clamp = p.has_max_val && p.N > 0;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x)
        evaporate_record(p, p.cells + (j << p.rec_shift), c, mx, clamp);
}

// Active-tile variant, two launches: (1) compact the ids of the tiles whose activity byte is set into a list,
// (2) one warp per listed 16x16 tile: all 8 record loads of a lane are issued before the first store; a tile whose
// cells all decayed to zero is retired.
__global__ void __launch_bounds__(256) k_tiles_compact(Params p, uint32_t *__restrict__ list) {
    const int64_t ntiles = (int64_t)p.E * p.tiles_x * p.tiles_y;
    const int lane = threadIdx.x & 31;
    for (int64_t t0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x - lane); t0 < ntiles;
         t0 += (int64_t)gridDim.x * blockDim.x) {
        const int64_t t = t0 + lane;
        const bool on = t < ntiles && p.tile_active[t] != 0;
        const unsigned m = __ballot_sync(0xffffffffu, on);
        if (m == 0) continue;
        unsigned long long basev = 0;
        if (lane == 0) basev = atomicAdd(p.tile_counter, (unsigned long long)__popc(m));
        basev = __shfl_sync(0xffffffffu, basev, 0);
        if (on) list[basev + __popc(m & ((1u << lane) - 1))] = (uint32_t)t;
    }
}
__global__ void __launch_bounds__(256) k_evaporate_tiles(Params p, const uint32_t *__restrict__ list) {
    const int lane = threadIdx.x & 31;
    const int64_t warp_g = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t n = (int64_t)*p.tile_counter;
    const int tiles_per_env = p.tiles_x * p.tiles_y;
    const double c = p.filt_center, mx = p.phero_max_val;
    const bool clamp = p.has_max_val && p.N > 0;
    for (int64_t idx = warp_g; idx < n; idx += nwarps) {
        const uint32_t tt = list[idx];
        const int e = (int)(tt / (uint32_t)tiles_per_env);
        const int tin = (int)(tt - (uint32_t)e * (uint32_t)tiles_per_env);
        const int tx = tin / p.tiles_y, ty = tin - tx * p.tiles_y;
        // a 16 x 16 tile is 2 x 2 blocks of 8 x 8 cells, each block 64 contiguous records: per pass the warp covers
        // half a block (32 records = 1 KB contiguous), every sector fully used
        bool any = false;
        const int bx0 = tx * 2, by0 = ty * 2;
        if (p.P == 2) {
            double2 v[8];
            uint8_t wl[8];
            uint8_t *rp[8];
#pragma unroll
            for (int pass = 0; pass < 8; ++pass) {
                int bx = bx0 + (pass >> 2);
                bx = bx < (p.Wp >> 3) ? bx : (p.Wp >> 3) - 1;                  // tiles past the map repeat the last block row
                const int by = by0 + ((pass >> 1) & 1);
                rp[pass] = rec_at(p, e, ((bx * p.nby + by) << 6) + (pass & 1) * 32 + lane);
                v[pass] = *reinterpret_cast<const double2 *>(rp[pass]);
                wl[pass] = rp[pass][p.wall_off] & 1;
            }
#pragma unroll
            for (int pass = 0; pass < 8; ++pass) {
                if (v[pass].x == 0.0 && v[pass].y == 0.0) continue;
                double a = wl[pass] ? 0.0 : v[pass].x * c, b = wl[pass] ? 0.0 : v[pass].y * c;
                a = a < 0.01 ? 0.0 : a;
                b = b < 0.01 ? 0.0 : b;
                if (clamp) { a = fmin(a, mx); b = fmin(b, mx); }
                *reinterpret_cast<double2 *>(rp[pass]) = make_double2(a, b);
                any |= (a != 0.0) || (b != 0.0);
            }
        } else {
#pragma unroll 1
            for (int pass = 0; pass < 8; ++pass) {
                const int bx = bx0 + (pass >> 2), by = by0 + ((pass >> 1) & 1);
                if (bx < (p.Wp >> 3))
                    any |= evaporate_record(p, rec_at(p, e, ((bx * p.nby + by) << 6) + (pass & 1) * 32 + lane), c, mx, clamp);
            }
        }
        if (!__any_sync(0xffffffffu, any) && lane == 0) p.tile_active[tt] = 0;
    }
}

// Diffusion stencil for DIFFUSE_FACTOR != 0 (pheromone.py:43-45: 3x3 convolution, boundary='fill', fillvalue=0, then
// the < 0.01 cut) with the wall zeroing of walls.py:30 applied to its inputs and the whole-plane clamp of
// pheromone.py:41.  One block = 64 x 64 outputs of one pheromone plane of one environment.  The (66 x 66) input tile
// with its halo arrives by ONE TMA tiled load (cp.async.bulk.tensor.3d, SASS UTMALDG) from the tensor map over the
// planes: the map's extents are the true (H, W), so everything outside the map -- the convolution's zero fill -- is
// filled with zeros by the TMA unit, also for negative coordinates; no bounds logic in the kernel.  Wall cells carry
// their flag in the sign bit: fmax(v, 0) is the zeroed input.  Output goes to the other plane, coalesced.
// (The innermost start coordinate of a tiled load must be 16-byte aligned -- an odd f64 coordinate is an illegal
// instruction, scripts/microbench/tma_probe.cu -- so the box starts two columns left of the tile: 66 x 68.)
// tile shape (measured on 1024 envs x 256^2, 2 pheromones, ms per update): 32x32 0.488, 16x64 0.474, 8x128 0.468,
// 64x32 0.407, 128x32 0.360, 64x64 0.354 (= 0.96 of the measured HBM copy peak)
constexpr int kStX = 64, kStY = 64, kStPadY = 2;
// Arithmetic: a warp owns 32 columns and a few consecutive output rows; a thread slides down its column
// keeping per input row the three clipped values (left, centre, right), their sum and the sum of the two sides, so an
// output costs 3 shared-memory loads and ~10 f64 operations instead of 9 and 27:
//     out = ring * (rowsum[x-1] + sides[x] + rowsum[x+1]) + centre_tap * v[x][y]
// (pheromone.py:7-9: the ring taps are all DIFFUSE_FACTOR (1 - EVAP), the centre is (1 - 8 DIFFUSE_FACTOR)(1 - EVAP);
// the summation order differs from scipy's, inside the 1e-5 bar, golden scenario `diffuse`).
__global__ void __launch_bounds__(256)
k_diffuse_tma(Params p, const __grid_constant__ CUtensorMap tmap, int src_z0, int nbx, int nby) {
    __shared__ __align__(128) double tile[kStX + 2][kStY + 2 + kStPadY];
    __shared__ __align__(8) unsigned long long bar;
    const int64_t ep = blockIdx.x / (nbx * nby);
    const int brem = (int)(blockIdx.x - ep * (nbx * nby));
    const int x0 = (brem / nby) * kStX, y0 = (brem % nby) * kStY;
    const uint32_t bar_s = (uint32_t)__cvta_generic_to_shared(&bar);
    const uint32_t tile_s = (uint32_t)__cvta_generic_to_shared(&tile[0][0]);
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_s) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        constexpr uint32_t bytes = (kStX + 2) * (kStY + 2 + kStPadY) * sizeof(double);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_s), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                     ::"r"(tile_s), "l"(&tmap), "r"(y0 - kStPadY), "r"(x0 - 1), "r"(src_z0 + (int)ep), "r"(bar_s) : "memory");
    }
    if (threadIdx.x == 0) {   // one thread polls the barrier (phase 0); the block barrier hands the tile to the others
        uint32_t done = 0;    // (all 256 threads polling cost 3/4 of the kernel's issue slots in ncu)
        while (!done)
            asm volatile("{\n .reg .pred q;\n mbarrier.try_wait.parity.shared::cta.b64 q, [%1], 0;\n selp.u32 %0, 1, 0, q;\n}"
                         : "=r"(done) : "r"(bar_s) : "memory");
    }
    __syncthreads();
    const double fc = p.filt_center, fr = p.filt_ring, mx = p.phero_max_val;
    const bool clamp = p.has_max_val && p.N > 0;
    constexpr int CG = kStY / 32;                      // column groups of 32 lanes
    constexpr int RPW = kStX * CG / 8;                 // output rows per warp (8 warps)
    const int warp = threadIdx.x >> 5, ly = (threadIdx.x & 31) + 32 * (warp % CG);
    const int gy = y0 + ly;
    const int lx0 = (warp / CG) * RPW;                 // first output row of this warp (tile row lx0 + 1)
    double *dst = p.phero_alt + ep * p.plane + gy;
    // tile column of (gy - 1): ly + kStPadY - 1
    const int c = ly + kStPadY - 1;
    double rs[RPW + 2], sd[RPW + 2], ce[RPW + 2];      // row sums, side sums, centres (raw centre keeps the wall sign)
#pragma unroll
    for (int r = 0; r < RPW + 2; ++r) {
        const double a = fmax(tile[lx0 + r][c], 0.0), raw = tile[lx0 + r][c + 1], b2 = fmax(tile[lx0 + r][c + 2], 0.0);
        const double m = fmax(raw, 0.0);
        sd[r] = a + b2;
        rs[r] = sd[r] + m;
        ce[r] = raw;
    }
    if (gy < p.H) {
#pragma unroll
        for (int r = 0; r < RPW; ++r) {
            const int gx = x0 + lx0 + r;
            if (gx >= p.W) break;
            double acc = (rs[r] + sd[r + 1] + rs[r + 2]) * fr + fmax(ce[r + 1], 0.0) * fc;
            acc = acc < 0.01 ? 0.0 : acc;
            if (clamp) acc = fmin(acc, mx);
            dst[(int64_t)gx * p.Hp] = signbit(ce[r + 1]) ? -acc : acc;
        }
    }
}
// Bits of an import's flag word (`bad`, the scratch word after the imported data), which ants_import_env_state
// returns as ANTS_E_ARG once the window's import has run:
//   kBadNonFinite  a pheromone or food value is NaN or +-inf (k_pack_f64): a deposit's fmin would turn a NaN into a
//                  saturated deposit, a NaN record reads as the boxed deposit of update 0, and the reference's
//                  convolution spreads the NaN to the neighbours -- not emulated
//   kBadAboveMax   lazy mode with max_val: a pheromone value above max_val (k_pack_f64).  The reference clamps it inside
//                  the next update, after evaporation (pheromone.py:41 after :44-45); a plain lazy record cannot, and
//                  the reference's own updates never leave such a value (each one clamps the whole plane)
//   kBadNegative   diffusion: a negative or NaN plane value (k_plane_walls); its sign bit would be read as the wall flag
constexpr uint32_t kBadNonFinite = 1u, kBadAboveMax = 2u, kBadNegative = 4u;
// after an import: the sign bit of every plane value = the wall bit of its cell record.  `bad` is non-null when the
// planes were just imported, so they still hold the caller's values.
__global__ void k_plane_walls(Params p, int env0, int n_env, uint32_t *bad) {
    const int64_t n = (int64_t)n_env * p.W * p.H;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
        int64_t ex = j / p.H;
        int y = (int)(j - ex * p.H);
        int64_t e = ex / p.W;
        int x = (int)(ex - e * p.W);
        e += env0;
        const bool wall = ld_wall(p, rec_at(p, (int)e, cidx(p, x, y)));
        for (int k = 0; k < p.P; ++k) {
            double *pv = plane_at(p, (int)e, k, x, y);
            const double v = *pv, a = fabs(v);
            if (bad != nullptr && !(v >= 0.0)) atomicOr(bad, kBadNegative);
            *pv = wall ? -a : a;
        }
    }
}

// Ants.emit_pheromones -> Pheromone.add_pheromones (ants.py:98-100, pheromone.py:36-41): the owner of each cell
// adds its activation and clamps to max_val.
__global__ void __launch_bounds__(256) k_deposit_commit(Params p, uint32_t owner_stamp, uint32_t now, uint32_t now_abs) {
    pdl_begin();
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.EN) return;
    int e = (int)(i / p.N);
    int a = (int)(i - (int64_t)e * p.N);
    int cx = cell_of(p.x[i], p.W), cy = cell_of(p.y[i], p.H);
    int cell = cidx(p, cx, cy);
    if (p.owner[(int64_t)e * p.plane + cell] != (owner_stamp | (uint32_t)a)) return;
    if (p.diffuse) {                                                           // planes: magnitude = value, sign = wall
        for (int k = 0; k < p.P; ++k) {
            const double av = p.act[(int64_t)k * p.EN + i];
            if (av == 0.0) continue;
            double *pv = plane_at(p, e, k, cx, cy);
            const double old = *pv;
            double v = fabs(old) + av;
            if (p.has_max_val) v = fmin(v, p.phero_max_val);
            *pv = signbit(old) ? -v : v;
        }
        return;
    }
    uint8_t *r = rec_at(p, e, cell);
    bool wrote = false;
    for (int k = 0; k < p.P; ++k) {
        double av = p.act[(int64_t)k * p.EN + i];
        if (av == 0.0) continue;
        double v = phero_value(p, r, k, now, now_abs) + av;                    // (lazy: evaporated up to this update)
        if (p.has_max_val) v = fmin(v, p.phero_max_val);
        phero_store(p, r, k, v, now, now_abs);
        wrote = true;
    }
    if (wrote && p.tile_active != nullptr)
        p.tile_active[((int64_t)e * p.tiles_x + cx / kTile) * p.tiles_y + cy / kTile] = 1;
}

// Anthill.update as a sweep over the disc's bounding box (first update after an import, quirk Q10).
__global__ void __launch_bounds__(256) k_absorb_sweep(Params p) {
    __shared__ double red[256];
    int e = blockIdx.x;
    const int32_t *hl = p.hill + 4 * e;
    int r = hl[2];
    int x0 = max(hl[0] - r, 0), x1 = min(hl[0] + r, p.W - 1);
    int y0 = max(hl[1] - r, 0), y1 = min(hl[1] + r, p.H - 1);
    int bw = x1 - x0 + 1, bh = y1 - y0 + 1;
    double acc = 0.0;
    if (bw > 0 && bh > 0) {
        for (int t = threadIdx.x; t < bw * bh; t += blockDim.x) {
            int cx = x0 + t / bh, cy = y0 + t % bh;
            if (!in_hill(hl, cx, cy)) continue;
            uint8_t *fr = rec_at(p, e, cidx(p, cx, cy));
            double v = ld_food(p, fr);
            if (v != 0.0) { acc += v; st_food(p, fr, v - v); }
        }
    }
    red[threadIdx.x] = acc;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0 && red[0] != 0.0) p.hill_food[e] += red[0];
}

// ------------------------------------------------------------------------------------------------ import / export helpers
// dense host-layout arrays <-> record fields.  `dense` is [E][planes_per_env][W][H]; field = plane `k` of them.
// `bad`: the import's flag word (kBad* above).
__global__ void k_pack_f64(Params p, const double *__restrict__ dense, int planes_per_env, int k, int byte_off,
                           int phero_k, uint32_t now, uint32_t now_abs, int env0, int n_env, uint32_t *bad) {
    const int64_t n = (int64_t)n_env * p.W * p.H;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
        int64_t ex = j / p.H;
        int y = (int)(j - ex * p.H);
        int64_t e = ex / p.W;                                                  // position in the imported window
        int x = (int)(ex - e * p.W);
        double v = dense[((e * planes_per_env + k) * p.W + x) * p.H + y];
        if (!isfinite(v)) atomicOr(bad, kBadNonFinite);
        else if (phero_k >= 0 && p.lazy && p.has_max_val && v > p.phero_max_val) atomicOr(bad, kBadAboveMax);
        e += env0;
        uint8_t *r = rec_at(p, (int)e, cidx(p, x, y));
        if (phero_k >= 0 && p.diffuse) {
            *plane_at(p, (int)e, phero_k, x, y) = v;                           // (k_plane_walls sets the sign afterwards)
        } else if (phero_k >= 0) {
            phero_store(p, r, phero_k, v, now, now_abs);
        } else {
            st_food(p, r, v);
        }
    }
}
// export of the envs [env0, env0 + n_env): dense arrays are indexed by the env's position in that window
__global__ void k_unpack_f64(Params p, double *__restrict__ dense, int planes_per_env, int k, int byte_off,
                             int phero_k, uint32_t now, uint32_t now_abs, int env0, int n_env) {
    const int64_t n = (int64_t)n_env * p.W * p.H;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
        int64_t ex = j / p.H;
        int y = (int)(j - ex * p.H);
        int64_t el = ex / p.W;
        int x = (int)(ex - el * p.W);
        const int e = env0 + (int)el;
        uint8_t *r = rec_at(p, e, cidx(p, x, y));
        double v = phero_k >= 0 ? (p.diffuse ? plane_value(p, e, phero_k, x, y) : phero_value(p, r, phero_k, now, now_abs))
                                : ld_food(p, r);
        dense[((el * planes_per_env + k) * p.W + x) * p.H + y] = v;
    }
}
// what: 0 = walls (stored as 0/1), 1 = explored (meta low half: 0xFFFF = explored long ago; occupancy cleared)
__global__ void k_pack_u8(Params p, const uint8_t *__restrict__ dense, int what, int env0, int n_env) {
    const int64_t n = (int64_t)n_env * p.W * p.H;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
        int64_t ex = j / p.H;
        int y = (int)(j - ex * p.H);
        int64_t e = ex / p.W;
        int x = (int)(ex - e * p.W);
        uint8_t *r = rec_at(p, env0 + (int)e, cidx(p, x, y));
        if (what == 0) st_wall(p, r, dense[j] != 0);
        else { st_explored(p, r, dense[j] ? p.explored_old : 0u); st_occ(p, r, 0u); }
    }
}
__global__ void k_unpack_u8(Params p, uint8_t *__restrict__ dense, int what, int env0, int n_env) {
    const int64_t n = (int64_t)n_env * p.W * p.H;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
        int64_t ex = j / p.H;
        int y = (int)(j - ex * p.H);
        int64_t el = ex / p.W;
        int x = (int)(ex - el * p.W);
        uint8_t *r = rec_at(p, env0 + (int)el, cidx(p, x, y));
        dense[j] = what == 0 ? (ld_wall(p, r) ? 1 : 0) : (ld_explored(p, r) ? 1 : 0);
    }
}
// the anthill disc as a bit of every cell record (anthill.py:31-33), after the anthill was imported
__global__ void k_hill_mark(Params p, int env0, int n_env) {
    const int64_t n = (int64_t)n_env * p.W * p.H;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
        int64_t ex = j / p.H;
        int y = (int)(j - ex * p.H);
        int64_t e = ex / p.W;
        int x = (int)(ex - e * p.W);
        e += env0;
        st_hill(p, rec_at(p, (int)e, cidx(p, x, y)), in_hill(p.hill + 4 * e, x, y));
    }
}
// generation counters are 16 bit: before one wraps, fold every live stamp into the "long ago" value
__global__ void k_meta_renormalize(Params p, int fold_explored, int clear_occ) {
    int64_t n = (int64_t)p.E * p.plane;
    if (p.rec8) {   // two 8-byte records per 128-bit access; the stamps are the high halves of words 1 and 3
        uint4 *recs = reinterpret_cast<uint4 *>(p.cells);
        for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n / 2; j += (int64_t)gridDim.x * blockDim.x) {
            uint4 v = recs[j];
            auto fix = [&](uint32_t w) -> uint32_t {
                uint32_t occ = (w >> 16) & 0xFFu, ex = w >> 24;               // [hill|occ_gen], [wall|explored_gen]
                if (fold_explored) { const uint32_t g = ex & 0x7Fu; if (g != 0u && g != 0x7Fu) ex |= 0x7Fu; }
                if (clear_occ) occ &= 0x80u;
                return (w & 0xFFFFu) | (occ << 16) | (ex << 24);
            };
            const uint32_t y = fix(v.y), w = fix(v.w);
            if (y != v.y || w != v.w) { v.y = y; v.w = w; recs[j] = v; }
        }
        return;
    }
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
        uint8_t *r = p.cells + (j << p.rec_shift);
        if (fold_explored) { uint32_t g = ld_explored(p, r); if (g != 0u && g != p.explored_old) st_explored(p, r, p.explored_old); }
        if (clear_occ && ld_occ(p, r) != 0u) st_occ(p, r, 0u);
    }
}
// lazy mode: re-base every PLAIN pheromone value to timestamp 0 (before the small counter wraps); boxed saturated
// deposits are left alone unless `unbox` is set (the 22-bit absolute counter is about to wrap)
__global__ void k_lazy_fold(Params p, uint32_t now, uint32_t now_abs, int unbox) {
    if (!unbox && *p.plain_flag == 0u) return;         // only saturated (boxed) deposits exist: nothing to re-base
    int64_t n = (int64_t)p.E * p.plane;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
        uint8_t *r = p.cells + (j << p.rec_shift);
        for (int k = 0; k < p.P; ++k) {
            bool boxed, zero;
            if (p.rec8) {
                // expired boxed deposits are cleared when `unbox` is set (the 15-bit step would alias); plain values
                // are re-based to timestamp 0 in their side slots
                const uint32_t c = reinterpret_cast<const uint16_t *>(r)[k];
                if (c == 0u) continue;
                if (c & kBox8) {
                    if (unbox && ((now_abs - c) & kBox8Mask) >= (uint32_t)p.tab_len) reinterpret_cast<uint16_t *>(r)[k] = 0;
                    continue;
                }
                const double v = phero_value(p, r, k, now, now_abs);
                if (v == 0.0) { reinterpret_cast<uint16_t *>(r)[k] = 0; continue; }
                p.side_val[rec8_index(p, r) * 3 + k] = (float)v;
                rec_set_ts(p, r, k, 0u);
                continue;
            }
            if (p.rec16) { uint32_t b = reinterpret_cast<const uint32_t *>(r)[k]; boxed = is_boxed32(b); zero = b == 0u; }
            else { unsigned long long b = reinterpret_cast<const unsigned long long *>(r)[k]; boxed = is_boxed64(b); zero = b == 0ull; }
            if (zero || (boxed && !unbox)) { if (!boxed) rec_set_ts(p, r, k, 0u); continue; }
            const double v = phero_value(p, r, k, now, now_abs);
            // written as a plain number valid at timestamp 0 (never re-boxed: it is no longer max_val unless age 0)
            if (p.rec16) reinterpret_cast<float *>(r)[k] = (float)v; else reinterpret_cast<double *>(r)[k] = v;
            rec_set_ts(p, r, k, 0u);
            // an unboxed deposit is a plain value like any other: the row perception kernel decodes plain values and
            // later folds re-base them only while the flag is set
            if (boxed && v != 0.0 && *p.plain_flag == 0u) *p.plain_flag = 1u;
        }
    }
}
__global__ void k_rock_grid_build(Params p, int env0) {   // one block per imported env
    const int e = env0 + blockIdx.x;
    const int gcells = p.grid_w * p.grid_h;
    unsigned long long *g = p.rock_grid + (int64_t)e * gcells;
    for (int k = threadIdx.x; k < gcells; k += blockDim.x) g[k] = 0ull;
    __syncthreads();
    for (int r = threadIdx.x; r < p.R; r += blockDim.x)
        rock_grid_mark(p, e, r, p.rock_c[((int64_t)e * p.R + r) * 2], p.rock_c[((int64_t)e * p.R + r) * 2 + 1],
                       p.rock_rad[(int64_t)e * p.R + r]);
}
__global__ void k_tiles_from_phero(Params p, int env0, int n_env) {
    // mark every tile that holds a non-zero pheromone cell (after import)
    const int64_t tiles_per_env = (int64_t)p.tiles_x * p.tiles_y;
    const int64_t ntiles = (int64_t)n_env * tiles_per_env;
    for (int64_t tw = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; tw < ntiles; tw += (int64_t)gridDim.x * blockDim.x) {
        const int64_t t = tw + (int64_t)env0 * tiles_per_env;
        int e = (int)(t / tiles_per_env);
        int tin = (int)(t - (int64_t)e * tiles_per_env);
        int tx = tin / p.tiles_y, ty = tin - tx * p.tiles_y;
        bool any = false;
        for (int dx = 0; dx < kTile && !any; ++dx) {
            int row = tx * kTile + dx;
            if (row >= p.W) break;
            for (int dy = 0; dy < kTile && !any; ++dy) {
                uint8_t *r = rec_at(p, e, cidx(p, row, ty * kTile + dy));
                for (int k = 0; k < p.P; ++k) any |= *rec_phero(r, k) != 0.0;
            }
        }
        p.tile_active[t] = any ? 1 : 0;
    }
}

}  // namespace ants

#include "ants_perceive_rows.cuh"
#include "ants_env_fused.cuh"
