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


def wald_f32(w1, w2, w3, mean, scale):
    """sample_distance_f32 for the Wald (numpy legacy): with Y = mean z^2 (z = normal_f32(w1, w2)),
    X = mean + mean / (2 scale) (Y - sqrtf(4 scale Y + Y^2)), U = uniform_f32(w3), the distance is X when
    U <= mean / (mean + X) and mean^2 / X otherwise.  Returns (distance in float64, relative bound,
    ambiguous): `ambiguous` flags the draws whose U lies within the bound of the threshold, where the
    device may take the other branch.  The subtraction Y - sqrt(...) cancels for large Y; the bound
    carries the float32 roundings of Y and of the square root through it."""
    assert float(np.float32(mean)) == mean and float(np.float32(scale)) == scale, 'use float32-exact parameters'
    mu_2l = float(np.float32(mean) / (np.float32(2.0) * np.float32(scale)))     # the device's float32 value
    z, e_z = normal_f32(w1, w2)
    Y = mean * z * z
    e_Y = mean * (2 * np.abs(z) * e_z + e_z * e_z) + Y * 2 * _F32
    S = 4 * scale * Y + Y * Y
    e_S = (4 * scale + 2 * Y + e_Y) * e_Y + S * 3 * _F32
    R = np.sqrt(S)
    e_R = np.minimum(np.sqrt(e_S), e_S / np.maximum(2 * R, 1e-300)) + R * _F32
    D = Y - R
    e_D = e_Y + e_R + np.abs(D) * _F32
    X = mean + mu_2l * D
    e_X = mu_2l * e_D + (np.abs(mu_2l * D) + np.abs(X)) * _F32
    U = uniform_f32(w3).astype(np.float64)
    T = mean / (mean + X)
    e_T = T * (e_X / np.abs(mean + X) + 2 * _F32)
    first = U <= T
    with np.errstate(divide='ignore', invalid='ignore'):
        d = np.where(first, X, mean * mean / X)
        rel = np.where(first, e_X / X, e_X / X + 2 * _F32)
    ambiguous = (np.abs(U - T) <= e_T) | ~(rel < 0.01)        # near the threshold, or X not resolved
    return d, rel, ambiguous


# ---- the on-the-fly conductance-surface direction (gnx_kernels.cuh vonmises_tab, surface_direction_from_neigh) ----
VM_TAB_CELLS, VM_TAB_FINE = 4096, 256
VM_TAB_LEN = VM_TAB_CELLS + 1 + VM_TAB_FINE + 1
PI_F = np.float32(3.14159265358979)
# the directions of the 8 queen neighbours in row-major order, as the device's float32 constants
SURF_DIRS = np.array([np.float32(-3) * PI_F / np.float32(4), -PI_F / np.float32(2), -PI_F / np.float32(4), PI_F,
                      np.float32(0), np.float32(3) * PI_F / np.float32(4), PI_F / np.float32(2), PI_F / np.float32(4)],
                     dtype=np.float32)


def _round_f32(q):
    """A Fraction rounded to the nearest float32, ties to even."""
    from fractions import Fraction
    x = np.float32(float(q))
    best = None
    for c in (np.nextafter(x, np.float32(-np.inf)), x, np.nextafter(x, np.float32(np.inf))):
        d = abs(Fraction(float(c)) - q)
        if best is None or d < best[0] or (d == best[0] and (int(np.float32(c).view(np.uint32)) & 1) == 0):
            best = (d, c)
    return np.float32(best[1])


def fma_f32(a, b, c):
    """fmaf(a, b, c) on float32 arrays: a b is exact in float64; when the float64 sum s = a b + c is exact
    too (TwoSum error term zero) it is rounded to float32 once.  Otherwise s differs from the exact sum x,
    and rounding s to float32 can only go wrong when s sits exactly on a float32 midpoint (midpoints are
    float64 numbers and rounding to float64 is monotone, so x and s lie strictly on the same side of every
    other midpoint); those sums are rounded from a Fraction of the exact value."""
    from fractions import Fraction
    a, b, c = np.broadcast_arrays(*(np.atleast_1d(np.asarray(v, dtype=np.float32)) for v in (a, b, c)))
    p = a.astype(np.float64) * b.astype(np.float64)
    cc = np.broadcast_to(c.astype(np.float64), p.shape)
    s = p + cc
    bp = s - p
    err = (p - (s - bp)) + (cc - bp)
    out = np.asarray(s.astype(np.float32))
    s32 = out.astype(np.float64)
    nb = np.nextafter(out, np.where(s > s32, np.float32(np.inf), np.float32(-np.inf)).astype(np.float32))
    mid = (s != s32) & (s == (s32 + nb.astype(np.float64)) / 2)
    for i in zip(*np.nonzero((err != 0) & mid)):
        out[i] = _round_f32(Fraction(float(p[i])) + Fraction(float(cc[i])))
    return out


def vonmises_tab(r, tab):
    """vonmises_tab for kappa >= 1e-8 from the word r: float32 |theta| interpolated in the quantile table,
    negated when bit 31 is set."""
    r = np.asarray(r, dtype=np.uint32)
    tab = np.asarray(tab, dtype=np.float32)
    v = (r << np.uint32(1)).astype(np.uint32)
    k = (v >> np.uint32(20)).astype(np.int64)
    coarse = k < VM_TAB_CELLS - 1
    k2 = ((v >> np.uint32(12)) & np.uint32(0xff)).astype(np.int64)
    f = np.where(coarse, ((v >> np.uint32(1)) & np.uint32(0x7ffff)).astype(np.float32) * np.float32(1.0 / 524288.0),
                 ((v >> np.uint32(1)) & np.uint32(0x7ff)).astype(np.float32) * np.float32(1.0 / 2048.0))
    ia = np.where(coarse, k, VM_TAB_CELLS + 1 + k2)
    a, b = tab[ia], tab[ia + 1]
    res = fma_f32(f, b - a, a)
    return np.where((r >> np.uint32(31)) != 0, -res, res)


def surface_direction(words, k, nv, mixture, kappa, tab):
    """surface_direction_from_neigh in float32 for each row: the neighbourhood nv (float32[n, 8], row-major
    queen neighbours of the zero-embedded raster), the stream's words from column k (int or int[n]).
    Returns (float16 direction, number of words used): the mixture draw (one uniform_f32 word) when
    `mixture`, then one von Mises word (the table word, or a uniform_f32 word when kappa < 1e-8)."""
    words = np.asarray(words, dtype=np.uint32)
    nv = np.asarray(nv, dtype=np.float32)
    n = nv.shape[0]
    rows = np.arange(n)
    k = np.broadcast_to(np.asarray(k, dtype=np.int64), (n,))
    s = np.zeros(n, np.float32)
    for j in range(8):
        s = s + nv[:, j]
    if mixture:
        pos = s > 0
        target = uniform_f32(words[rows, k]) * np.where(pos, s, np.float32(8))
        acc = np.zeros(n, np.float32)
        loc = np.full(n, SURF_DIRS[7], np.float32)
        found = np.zeros(n, bool)
        for j in range(8):
            acc = acc + np.where(pos, nv[:, j], np.float32(1))
            hit = ~found & (target < acc)
            loc[hit] = SURF_DIRS[j]
            found |= hit
        kv = k + 1
    else:
        mx = nv.max(axis=1)
        sacc = np.zeros(n, np.float32)
        cnt = np.zeros(n, np.float32)
        for j in range(8):
            m = nv[:, j] == mx
            sacc = np.where(m, sacc + SURF_DIRS[j], sacc)
            cnt = cnt + m.astype(np.float32)
        loc = sacc / cnt
        kv = k
    wv = words[rows, kv]
    if np.float32(kappa) < np.float32(1e-8):
        vm = PI_F * (np.float32(2) * uniform_f32(wv) - np.float32(1))
    else:
        vm = vonmises_tab(wv, tab)
    v = (loc + vm).astype(np.float32)
    v = np.where(v >= PI_F, v - np.float32(2) * PI_F, np.where(v < -PI_F, v + np.float32(2) * PI_F, v))
    return v.astype(np.float32).astype(np.float16), (kv - k + 1)
