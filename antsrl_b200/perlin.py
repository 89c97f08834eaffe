"""Perlin walls for the map interface (SURVEY.md section 8-f, row 1).

The reference's default walls generator (`generator/map_generators.py:9-25`) thresholds
`utils.perlin_noise_generator` (`utils.py:7-18`), which calls `noise.pnoise2` of the third-party C extension
`noise` (caseman/noise; imported at `utils.py:2`, no version pinned anywhere in the reference, latest release
1.2.2) once per map cell.  That package is neither vendored in the reference nor installed here, and the
reference holds no test or golden vector for it, so this restatement of the package's published algorithm
(`_perlin.c`: `noise2` = Ken Perlin's improved gradient noise on the classic 256-entry permutation with the
12 + 4 edge gradients, single precision; `pnoise2` = the octave sum normalised by the amplitude sum) is
**parity unpinned**: it is checked by known-answer properties of the algorithm (zero on the integer lattice,
bounds, smoothness, period), not against outputs of the package.  It only shapes the walls bitmap, an input
of the step loop; it runs on the host, once per episode, vectorised over the whole map.  The device computes the same
float32 field bit for bit (antsrl_b200/csrc/ants_perlin.cuh): `perlin_noise_device`, and the Perlin layers of
`BatchedAnts.generate_env_maps` that `BatchedEnvironmentGenerator.reset(..., perlin="device")` writes.
"""
import collections
import ctypes as C
import random

import numpy as np

_PERM = np.array([
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
    78, 66, 215, 61, 156, 180], dtype=np.int64)
_PERM = np.concatenate([_PERM, _PERM])          # the package stores the period twice: PERM[A + j] needs no wrap
# x and y components of the package's GRAD3 table (12 cube-edge gradients + 4 repeats)
_GX = np.array([1, -1, 1, -1, 1, -1, 1, -1, 0, 0, 0, 0, 1, -1, 0, 0], dtype=np.float32)
_GY = np.array([1, 1, -1, -1, 0, 0, 0, 0, 1, -1, 1, -1, 0, 0, -1, 1], dtype=np.float32)

_F = np.float32


def _grad2(h, x, y):
    h = h & 15
    return x * _GX[h] + y * _GY[h]


def _lerp(t, a, b):
    return a + t * (b - a)


def noise2(x, y, repeatx=1024.0, repeaty=1024.0, base=0):
    """One octave of 2-D improved Perlin noise, float32 arrays in, float32 out (the package's `noise2`)."""
    x = np.asarray(x, dtype=_F)
    y = np.asarray(y, dtype=_F)
    repeatx, repeaty = _F(repeatx), _F(repeaty)
    i = np.floor(np.fmod(x, repeatx)).astype(np.int64)
    j = np.floor(np.fmod(y, repeaty)).astype(np.int64)
    ii = np.fmod((i + 1).astype(_F), repeatx).astype(np.int64)      # (int) truncates
    jj = np.fmod((j + 1).astype(_F), repeaty).astype(np.int64)
    i = (i & 255) + base
    j = (j & 255) + base
    ii = (ii & 255) + base
    jj = (jj & 255) + base
    x = x - np.floor(x)
    y = y - np.floor(y)
    fx = x * x * x * (x * (x * _F(6) - _F(15)) + _F(10))
    fy = y * y * y * (y * (y * _F(6) - _F(15)) + _F(10))
    A = _PERM[i]
    AA = _PERM[A + j]
    AB = _PERM[A + jj]
    B = _PERM[ii]
    BA = _PERM[B + j]
    BB = _PERM[B + jj]
    one = _F(1)
    return _lerp(fy, _lerp(fx, _grad2(_PERM[AA], x, y), _grad2(_PERM[BA], x - one, y)),
                 _lerp(fx, _grad2(_PERM[AB], x, y - one), _grad2(_PERM[BB], x - one, y - one))).astype(_F)


def pnoise2(x, y, octaves=1, persistence=0.5, lacunarity=2.0, repeatx=1024.0, repeaty=1024.0, base=0):
    """`noise.pnoise2`: fractal sum of `octaves` octaves, divided by the sum of the amplitudes."""
    if octaves < 1:
        raise ValueError("Expected octaves value > 0")
    x = np.asarray(x, dtype=_F)
    y = np.asarray(y, dtype=_F)
    if octaves == 1:
        return noise2(x, y, repeatx, repeaty, base)
    freq, amp, mx = _F(1), _F(1), _F(0)
    total = np.zeros(np.broadcast(x, y).shape, dtype=_F)
    for _ in range(octaves):
        total = total + noise2(x * freq, y * freq, _F(repeatx) * freq, _F(repeaty) * freq, base) * amp
        mx = mx + amp
        freq = freq * _F(lacunarity)
        amp = amp * _F(persistence)
    return (total / mx).astype(_F)


def perlin_noise_generator(w, h, offset_x, offset_y, scale=22.0, octaves=2, persistence=0.5, lacunarity=2.0):
    """utils.py:7-18: gen[i][j] = pnoise2((i + offset_x) / scale, (j + offset_y) / scale, ...), float64 (w, h)."""
    xs = ((np.arange(w) + offset_x) / scale).astype(_F)[:, None]     # the division is Python's (double), the call
    ys = ((np.arange(h) + offset_y) / scale).astype(_F)[None, :]     # narrows its arguments to C floats
    xs, ys = np.broadcast_arrays(xs, ys)
    return pnoise2(xs, ys, octaves=octaves, persistence=persistence, lacunarity=lacunarity, base=0).astype(np.float64)


# A Perlin map layer in the form ants_generate_env_maps_ex takes (AntsPerlinLayer): offsets (n, 2) int32 of n envs, and
# the generator's parameters, shared by the envs
PerlinLayer = collections.namedtuple("PerlinLayer", "offsets scale density octaves persistence lacunarity")


def perlin_layer_struct(layer):
    """-> (AntsPerlinLayer, the contiguous int32 offsets it points to: keep it alive for the call)."""
    from ._cabi import AntsPerlinLayer
    offs = np.ascontiguousarray(layer.offsets, dtype=np.int32)
    if offs.ndim != 2 or offs.shape[1] != 2:
        raise ValueError("Perlin offsets must have shape (n, 2); got %r" % (offs.shape,))
    s = AntsPerlinLayer()
    s.offsets = offs.ctypes.data_as(C.POINTER(C.c_int32))
    s.scale, s.density = float(layer.scale), float(layer.density)
    s.octaves, s.reserved = int(layer.octaves), 0
    s.persistence, s.lacunarity = float(layer.persistence), float(layer.lacunarity)
    return s, offs


def perlin_noise_device(w, h, offsets, scale=22.0, octaves=2, persistence=0.5, lacunarity=2.0, device=0):
    """`perlin_noise_generator` on the GPU (ants_perlin_noise) for n offset pairs at once: offsets (n, 2) of
    (offset_x, offset_y) -> float32 CUDA tensor (n, w, h), equal bit for bit to
    ``perlin_noise_generator(w, h, ox, oy, ...).astype(np.float32)`` (the host function widens its float32 field to
    float64).  The same device code writes the Perlin layers of `BatchedAnts.generate_env_maps`."""
    import torch
    from ._cabi import check, load_library
    lib = load_library()
    layer, offs = perlin_layer_struct(PerlinLayer(offsets, scale, 0.0, octaves, persistence, lacunarity))
    dev = torch.device("cuda", device)
    out = torch.empty((offs.shape[0], int(w), int(h)), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream().cuda_stream
        check(lib, lib.ants_perlin_noise(int(device), C.byref(layer), offs.shape[0], int(w), int(h),
                                         C.c_void_p(out.data_ptr()), C.c_void_p(stream)))
    return out


class PerlinGenerator:
    """map_generators.py:9-25: walls where the noise exceeds `density`; draws the two offsets from the global
    `random` module exactly like the reference (so the draws that follow it stay aligned)."""

    def __init__(self, scale=22.0, density=0.05, octaves=2, persistence=0.5, lacunarity=2.0):
        self.scale, self.density, self.octaves = scale, density, octaves
        self.persistence, self.lacunarity = persistence, lacunarity

    def draw_offsets(self):
        """-> int32 (offset_x, offset_y): exactly the two `random.randint` calls of `generate`, in its order."""
        offset_x = random.randint(-10000, 10000)
        offset_y = random.randint(-10000, 10000)
        return np.array([offset_x, offset_y], dtype=np.int32)

    def stamp(self, w, h, offsets):
        """bool (w, h): the map of the drawn offsets, noise > density."""
        offset_x, offset_y = (int(v) for v in offsets)
        return perlin_noise_generator(w, h, offset_x=offset_x, offset_y=offset_y, scale=self.scale,
                                      octaves=self.octaves, persistence=self.persistence,
                                      lacunarity=self.lacunarity) > self.density

    def generate(self, w, h):
        return self.stamp(w, h, self.draw_offsets())

    def layer(self, offsets):
        """The PerlinLayer of this generator for the (n, 2) offsets of n envs (BatchedAnts.generate_env_maps)."""
        return PerlinLayer(np.asarray(offsets, dtype=np.int32).reshape(-1, 2), self.scale, self.density, self.octaves,
                           self.persistence, self.lacunarity)
