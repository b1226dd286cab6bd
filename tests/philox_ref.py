"""The device's counter-based random streams restated in numpy (gnx_common.cuh philox4x32_10 /
RngStream, gnx_kernels.cuh uniform_f32 / uniform_pos_f32 / normal_f32).

Every random number of a free-running step is a pure function of (seed, entity id, call site,
time step, word position), so the tests can rebuild the draws of any stage on the host and feed
them to the oracle's stage functions: the free-running path is then checked exactly, not only in
distribution.

A stream of (seed, id, site, t) is the sequence of Philox4x32-10 blocks with counter
(id_lo, id_hi ^ (site << 24), (uint32) t, block) and key (seed_lo, seed_hi), block = 0, 1, ...,
each block consumed as its words x, y, z, w."""
import numpy as np

M32 = np.uint64(0xFFFFFFFF)
_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)

# call sites (gnx_common.cuh)
SITE_MOVE, SITE_MATE, SITE_BIRTHS, SITE_GAMETE, SITE_DISP, SITE_SEX = 1, 2, 3, 4, 5, 6
SITE_DEATH, SITE_PANMIXIA, SITE_MUTATE, SITE_GENOME_INIT = 7, 8, 9, 10


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32 with 10 rounds on (broadcast) arrays of 32-bit values -> four uint32 arrays."""
    c = [np.asarray(v, dtype=np.uint64) & M32 for v in (c0, c1, c2, c3)]
    k0 = np.asarray(k0, dtype=np.uint64) & M32
    k1 = np.asarray(k1, dtype=np.uint64) & M32
    for _ in range(10):
        p0 = _M0 * c[0]                     # < 2^64: exact in uint64
        p1 = _M1 * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & M32]
        k0 = (k0 + _W0) & M32
        k1 = (k1 + _W1) & M32
    return tuple(v.astype(np.uint32) for v in c)


def stream_words(seed, ids, site, t, n_words):
    """uint32[len(ids), n_words]: the first n_words words of the stream of each id."""
    ids = np.atleast_1d(np.asarray(ids, dtype=np.int64)).astype(np.uint64)
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    lo = ids & M32
    hi = (ids >> np.uint64(32)) ^ np.uint64((int(site) << 24) & 0xFFFFFFFF)
    tt = np.uint64(int(t) & 0xFFFFFFFF)
    out = np.empty((len(ids), 4 * ((int(n_words) + 3) // 4)), dtype=np.uint32)
    for b in range(out.shape[1] // 4):
        x, y, z, w = philox4x32_10(lo, hi, tt, np.uint64(b), seed & 0xFFFFFFFF, seed >> 32)
        out[:, 4 * b:4 * b + 4] = np.stack([x, y, z, w], axis=1)
    return out[:, :n_words]


def uniform(words, k):
    """RngStream::uniform() from words k and k + 1: 53 bits, ((w_k >> 5) 2^26 + (w_k+1 >> 6)) / 2^53."""
    a = (words[:, k] >> np.uint32(5)).astype(np.float64)
    b = (words[:, k + 1] >> np.uint32(6)).astype(np.float64)
    return (a * 67108864.0 + b) / 9007199254740992.0


def uniform_f32(w):
    """[0, 1) in float32 from the top 24 bits of one word."""
    return (np.asarray(w, dtype=np.uint32) >> np.uint32(8)).astype(np.float32) * np.float32(1.0 / 16777216.0)


def uniform_pos_f32(w):
    """(0, 1] in float32: ((float) w + 1) 2^-32, each operation rounded to float32."""
    return (np.asarray(w, dtype=np.uint32).astype(np.float32) + np.float32(1.0)) * np.float32(1.0 / 4294967296.0)


def choose_k(R, n):
    """Uniform integer in [0, n) from a word: (R n) >> 32."""
    return ((np.asarray(R, dtype=np.uint64) * np.uint64(n)) >> np.uint64(32)).astype(np.int64)


# ---- the float32 samplers of movement and dispersal, restated in float64 with an error bound ----
_LOGF_ABS = 2.0 ** -21.41      # __logf on [0.5, 2]: absolute error (CUDA C Programming Guide, intrinsic functions)
_F32 = 2.0 ** -24              # one float32 rounding, relative
_SINCOSPIF = 2.0 ** -23        # cospif / sincospif: 1 ulp on values of magnitude <= 1 (absolute)
_EXPF = 2.0 ** -22             # expf: 2 ulp, relative


def direction_f32(w):
    """The free direction (kappa < 1e-8): sincospif(2 u - 1) with u = uniform_f32(w).  Returns
    (cos, sin) in float64 and the absolute error bound of each component on the device."""
    a = np.pi * (2.0 * uniform_f32(w).astype(np.float64) - 1.0)
    return np.cos(a), np.sin(a), np.full(len(a), _SINCOSPIF)


def normal_f32(w1, w2):
    """normal_f32: sqrtf(-2 __logf(u1)) cospif(2 u2) -> (z in float64, bound on |z_device - z|)."""
    u1 = uniform_pos_f32(w1).astype(np.float64)
    u2 = uniform_f32(w2).astype(np.float64)
    lg = np.log(u1)
    a = -2.0 * lg
    r = np.sqrt(a)
    c = np.cos(2.0 * np.pi * u2)
    z = r * c
    e_a = 2.0 * _LOGF_ABS * np.maximum(1.0, np.abs(lg))
    e_r = np.minimum(np.sqrt(e_a), e_a / np.maximum(2.0 * r, 1e-300)) + r * _F32
    e_z = e_r * np.abs(c) + (r + e_r) * _SINCOSPIF + np.abs(z) * 2 * _F32
    return z, e_z


def lognormal_f32(w1, w2, p1, p2):
    """sample_distance_f32 for the lognormal: expf((float) p1 + (float) p2 z) -> (distance, relative bound)."""
    assert float(np.float32(p1)) == p1 and float(np.float32(p2)) == p2, 'use float32-exact parameters'
    z, e_z = normal_f32(w1, w2)
    arg = p1 + p2 * z
    d = np.exp(arg)
    rel = abs(p2) * e_z + np.abs(arg) * 2 * _F32 + _EXPF
    return d, rel
