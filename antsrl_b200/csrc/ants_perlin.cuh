// ants_perlin.cuh -- sm_100a Perlin noise of the reference's default walls generator (PerlinGenerator,
// map_generators.py:9-25: utils.perlin_noise_generator over noise.pnoise2), bit for bit as antsrl_b200/perlin.py computes
// it.  One implementation serves k_reset_maps (walls / food of a new episode) and k_perlin_field (ants_perlin_noise).
//
// Exactness: perlin.py is float32 numpy, one rounding per product and sum, and the library is built with -fmad=false
// and IEEE division, so the device follows it operation by operation:
//   x = (float)((double)(cell + offset) / scale)                                  (Python's division, narrowed to float)
//   per octave: xf = x * freq, i = (int)floorf(fmodf(xf, rep)), ii = (int)fmodf((float)(i + 1), rep), both & 255,
//               f = xf - floorf(xf), fade = f*f*f*(f*(f*6-15)+10), lerp(t, a, b) = a + t*(b - a)
//   total = total + n*amp; mx = mx + amp; freq = freq*lac; amp = amp*pers; then total / mx (one octave: n itself)
// The gradients of GRAD3 are -1, 0 or 1, so their products are exact: they are selects, and x * 0 keeps numpy's sign of
// a zero product.  The host (ants_abi.cu, perlin_layer_check) rejects parameters whose integer parts leave int32.
#pragma once

namespace ants {

constexpr int kPerlinMaxOctaves = 32;
constexpr int kPerlinTile = 64;                // = kResetTile: the field kernel covers the tiles of k_reset_maps
constexpr int kPerlinThreads = 256;

// Ken Perlin's permutation (perlin.py _PERM); each CTA copies it, doubled, to shared memory (the lookups diverge)
__constant__ uint8_t kPerlinPerm[256] = {
    151, 160, 137, 91, 90, 15, 131, 13, 201, 95, 96, 53, 194, 233, 7, 225, 140, 36, 103, 30, 69, 142, 8, 99, 37, 240,
    21, 10, 23, 190, 6, 148, 247, 120, 234, 75, 0, 26, 197, 62, 94, 252, 219, 203, 117, 35, 11, 32, 57, 177, 33, 88,
    237, 149, 56, 87, 174, 20, 125, 136, 171, 168, 68, 175, 74, 165, 71, 134, 139, 48, 27, 166, 77, 146, 158, 231, 83,
    111, 229, 122, 60, 211, 133, 230, 220, 105, 92, 41, 55, 46, 245, 40, 244, 102, 143, 54, 65, 25, 63, 161, 1, 216,
    80, 73, 209, 76, 132, 187, 208, 89, 18, 169, 200, 196, 135, 130, 116, 188, 159, 86, 164, 100, 109, 198, 173, 186,
    3, 64, 52, 217, 226, 250, 124, 123, 5, 202, 38, 147, 118, 126, 255, 82, 85, 212, 207, 206, 59, 227, 47, 16, 58, 17,
    182, 189, 28, 42, 223, 183, 170, 213, 119, 248, 152, 2, 44, 154, 163, 70, 221, 153, 101, 155, 167, 43, 172, 9, 129,
    22, 39, 253, 19, 98, 108, 110, 79, 113, 224, 232, 178, 185, 112, 104, 218, 246, 97, 228, 251, 34, 242, 193, 238,
    210, 144, 12, 191, 179, 162, 241, 81, 51, 145, 235, 249, 14, 239, 107, 49, 192, 214, 31, 181, 199, 106, 157, 184,
    84, 204, 176, 115, 121, 50, 45, 127, 4, 150, 254, 138, 236, 205, 93, 222, 114, 67, 29, 24, 72, 243, 141, 128, 195,
    78, 66, 215, 61, 156, 180};

struct PerlinArgs {          // device form of AntsPerlinLayer
    const int2 *offsets;     // [n_env] (offset_x, offset_y); NULL: the layer is not Perlin
    double scale, density;
    int32_t octaves;
    float persistence, lacunarity;
};

struct PerlinSmem {
    int perm[512];
    float4 col[kPerlinTile];   // per octave: (x - floor x, fade, PERM[i], PERM[ii]) of each column of the tile
    float4 row[kPerlinTile];   // (y - floor y, fade, j, jj) of each row
};

// x * GX[h & 15] + y * GY[h & 15] of perlin.py
__device__ __forceinline__ float perlin_grad(int h, float x, float y) {
    h &= 15;
    const float gx = ((0x30FF >> h) & 1) ? (((0x20AA >> h) & 1) ? -x : x) : x * 0.f;
    const float gy = ((0xCF0F >> h) & 1) ? (((0x4A0C >> h) & 1) ? -y : y) : y * 0.f;
    return gx + gy;
}

// the axis terms of one coordinate c (already times freq) with the period rep = 1024 * freq: (frac, fade, i, ii)
__device__ __forceinline__ float4 perlin_axis(float c, float rep) {
    const int i = (int)floorf(fmodf(c, rep));
    const int ii = (int)fmodf((float)(i + 1), rep);
    const float f = c - floorf(c);
    return make_float4(f, f * f * f * (f * (f * 6.f - 15.f) + 10.f), __int_as_float(i & 255), __int_as_float(ii & 255));
}

// noise2 of perlin.py from a column's terms (x, fade x, A = PERM[i], B = PERM[ii]) and a row's (y, fade y, j, jj)
__device__ __forceinline__ float perlin_noise2(const int *perm, float4 c, float4 r) {
    const float x = c.x, y = r.x, fx = c.y, fy = r.y;
    const int A = __float_as_int(c.z), B = __float_as_int(c.w), j = __float_as_int(r.z), jj = __float_as_int(r.w);
    const float g_aa = perlin_grad(perm[perm[A + j]], x, y), g_ba = perlin_grad(perm[perm[B + j]], x - 1.f, y);
    const float g_ab = perlin_grad(perm[perm[A + jj]], x, y - 1.f), g_bb = perlin_grad(perm[perm[B + jj]], x - 1.f, y - 1.f);
    const float l0 = g_aa + fx * (g_ba - g_aa), l1 = g_ab + fx * (g_bb - g_ab);
    return l0 + fy * (l1 - l0);
}

// The thread's cells of a 64 x 64 tile, in the order of k_reset_maps' record pairs: pair i of thread t is the cells
// (lx, ly) and (lx, ly + 1) of the tile, lx = 8 i + (t >> 2 & 7), ly = 8 (t >> 5) + 2 (t & 3).
__device__ __forceinline__ int perlin_tile_lx(int i) { return (i << 3) + (((int)threadIdx.x >> 2) & 7); }
__device__ __forceinline__ int perlin_tile_ly() { return (((int)threadIdx.x >> 5) << 3) + (((int)threadIdx.x & 3) << 1); }

// pnoise2 at the thread's 2 * PAIRS cells of the tile at (x0, y0) of env el of the layer (v[2i], v[2i + 1]: pair i).
// Columns x >= W and rows y >= H take the coordinate of the last column / row of the map (their values are not used).
// Every thread of the CTA calls it: it synchronises.
template <int PAIRS>
__device__ void perlin_tile(PerlinSmem &s, const PerlinArgs &L, int el, int x0, int y0, int W, int H, float (&v)[2 * PAIRS]) {
    static_assert(PAIRS == kPerlinTile * kPerlinTile / 2 / kPerlinThreads, "two cells per pair, 256 threads a tile");
    const int t = (int)threadIdx.x;
    __syncthreads();                                         // (an earlier call may still read the tables)
    for (int k = t; k < 512; k += kPerlinThreads) s.perm[k] = kPerlinPerm[k & 255];
    // the scaled coordinate of column t (t < 64) or row t - 64 (t < 128): Python's double division, narrowed
    float base = 0.f;
    if (t < 2 * kPerlinTile) {
        const int2 off = L.offsets[el];
        const int c = t < kPerlinTile ? min(x0 + t, W - 1) + off.x : min(y0 + t - kPerlinTile, H - 1) + off.y;
        base = (float)((double)c / L.scale);
    }
    const float lac = L.lacunarity, pers = L.persistence;
    float freq = 1.f, amp = 1.f, mx = 0.f;
    const float zero = L.octaves == 1 ? -0.f : 0.f;          // -0 + n is n: one octave returns noise2 itself
#pragma unroll
    for (int k = 0; k < 2 * PAIRS; ++k) v[k] = zero;
    const int ly = perlin_tile_ly();
    for (int o = 0; o < L.octaves; ++o) {
        __syncthreads();                                     // the previous octave's terms are read
        if (t < 2 * kPerlinTile) {
            float4 a = perlin_axis(base * freq, 1024.f * freq);
            if (t < kPerlinTile) {
                a.z = __int_as_float(s.perm[__float_as_int(a.z)]);
                a.w = __int_as_float(s.perm[__float_as_int(a.w)]);
                s.col[t] = a;
            } else {
                s.row[t - kPerlinTile] = a;
            }
        }
        __syncthreads();
        const float4 r0 = s.row[ly], r1 = s.row[ly + 1];
#pragma unroll
        for (int i = 0; i < PAIRS; ++i) {
            const float4 c = s.col[perlin_tile_lx(i)];
            v[2 * i] = v[2 * i] + perlin_noise2(s.perm, c, r0) * amp;
            v[2 * i + 1] = v[2 * i + 1] + perlin_noise2(s.perm, c, r1) * amp;
        }
        mx = mx + amp;
        freq = freq * lac;
        amp = amp * pers;
    }
    if (L.octaves > 1) {
#pragma unroll
        for (int k = 0; k < 2 * PAIRS; ++k) v[k] = v[k] / mx;
    }
}

// ants_perlin_noise: the float32 field pnoise2 of n offset pairs, out [n][W][H]; one CTA per (env, 64 x 64 tile)
__global__ void __launch_bounds__(kPerlinThreads) k_perlin_field(PerlinArgs L, int W, int H, int tiles_y, int tiles,
                                                                 float *out) {
    __shared__ PerlinSmem s;
    constexpr int kPairs = kPerlinTile * kPerlinTile / 2 / kPerlinThreads;
    const int el = blockIdx.x / tiles, tt = blockIdx.x - el * tiles;
    const int x0 = tt / tiles_y * kPerlinTile, y0 = (tt % tiles_y) * kPerlinTile;
    float v[2 * kPairs];
    perlin_tile<kPairs>(s, L, el, x0, y0, W, H, v);
    const int y = y0 + perlin_tile_ly();
    float *const o = out + (int64_t)el * W * H;
#pragma unroll
    for (int i = 0; i < kPairs; ++i) {
        const int x = x0 + perlin_tile_lx(i);
        if (x >= W) continue;
        if (y < H) o[(int64_t)x * H + y] = v[2 * i];
        if (y + 1 < H) o[(int64_t)x * H + y + 1] = v[2 * i + 1];
    }
}

}  // namespace ants
