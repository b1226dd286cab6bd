"""Bit-packing of diploid genotypes and recombination paths (host-side, setup / API views).

Device layout (DESIGN.md): one row per individual = [homologue 0 | homologue 1], each
homologue padded to 128-bit units; locus l is bit (l % 32) of u32 word l // 32.  The
reference stores an (L, 2) int8 array per individual (structs/individual.py:102-106) and
recombination 'subsetters' as bitarrays of '10'/'01' units (structs/genome.py:209-226); the
packed path keeps only the homologue bit per locus.
"""
import numpy as np


def words_per_hap(L):
    return 4 * max(1, (int(L) + 127) // 128)


def pack_bits(bits):
    """bits uint8[..., nbits] (nbits multiple of 32) -> u32[..., nbits // 32], little-endian bits."""
    b = np.ascontiguousarray(bits, dtype=np.uint8)
    by = np.packbits(b, axis=-1, bitorder='little')
    return np.ascontiguousarray(by).view(np.uint32)


def pack_genomes(g):
    """int8[N, L, 2] -> u32[N, 2, W]."""
    g = np.asarray(g)
    n, L, _ = g.shape
    W = words_per_hap(L)
    bits = np.zeros((n, 2, W * 32), dtype=np.uint8)
    bits[:, :, :L] = np.transpose(g, (0, 2, 1))
    return pack_bits(bits).reshape(n, 2, W)


def unpack_genomes(packed, L):
    """u32[N, 2, W] -> int8[N, L, 2]."""
    packed = np.ascontiguousarray(packed, dtype=np.uint32)
    n = packed.shape[0]
    bits = np.unpackbits(packed.view(np.uint8).reshape(n, 2, 4 * packed.shape[2]), axis=-1, bitorder='little')
    return np.ascontiguousarray(np.transpose(bits[:, :, :L], (0, 2, 1))).astype(np.int8)


def pack_paths(paths):
    """uint8[n_paths, L] homologue index per locus -> u32[n_paths, W]."""
    paths = np.asarray(paths, dtype=np.uint8)
    n, L = paths.shape
    W = words_per_hap(L)
    bits = np.zeros((n, W * 32), dtype=np.uint8)
    bits[:, :L] = paths
    return pack_bits(bits).reshape(n, W)


def carrier_counts(n, p):
    """1-alleles per locus of a starting population of n individuals with allele frequencies p
    (genome.py:1108-1157): round(2n p) (numpy's half-to-even), one fewer where that makes a locus fixed
    although p < 1, one where it makes a locus lost although p > 0."""
    p = np.asarray(p, dtype=np.float64)
    c = np.round((2 * int(n)) * p, 0).astype(np.int64)
    c[(c == 2 * int(n)) & (p < 1)] -= 1
    c[(c == 0) & (p > 0)] = 1
    return c


def rows_to_loci(g_rows, nonneut_loci, L):
    """gen_arch.use_tskit = True (species.py:891-905): the reference's genotype arrays hold one ROW per
    non-neutral locus, int8[N, n_nonneut, 2].  The device keeps one bit per LOCUS: row r becomes locus
    nonneut_loci[r], neutral loci are zero."""
    g_rows = np.asarray(g_rows)
    g = np.zeros((g_rows.shape[0], int(L), 2), dtype=np.int8)
    g[:, np.asarray(nonneut_loci, dtype=np.int64), :] = g_rows
    return g


def loci_to_rows(g, nonneut_loci):
    """The reference's use_tskit = True view of by-locus genotypes: rows nonneut_loci, in order."""
    return np.ascontiguousarray(np.asarray(g)[:, np.asarray(nonneut_loci, dtype=np.int64), :])


# ---- column layout (gnx_create_cols): a use_tskit species' rows hold one column per non-neutral locus ----
MUT_MAX_NEW = 64          # GNX_MUT_MAX_NEW: non-neutral mutations one step may add at most


def col_capacity(n_nonneut):
    """Starting columns of a species with n_nonneut non-neutral loci: room for one step of new ones."""
    return 128 * ((int(n_nonneut) + MUT_MAX_NEW + 127) // 128)


def rows_to_cols(g_rows, col_locus, W):
    """int8[N, n_cols, 2] rows in ascending locus order (the reference's use_tskit Individual.g) -> u32[N, 2, W]
    column rows: bit j holds locus col_locus[j]."""
    g_rows = np.asarray(g_rows)
    col_locus = np.asarray(col_locus, dtype=np.int64)
    n = g_rows.shape[0]
    assert g_rows.shape[1] == len(col_locus), (g_rows.shape, len(col_locus))
    bits = np.zeros((n, 2, int(W) * 32), dtype=np.uint8)
    bits[:, :, np.argsort(col_locus, kind='stable')] = np.transpose(g_rows, (0, 2, 1))
    return pack_bits(bits).reshape(n, 2, int(W))


def cols_to_rows(packed, col_locus):
    """u32[N, 2, W] column rows -> int8[N, n_cols, 2] rows in ascending locus order."""
    order = np.argsort(np.asarray(col_locus, dtype=np.int64), kind='stable')
    return np.ascontiguousarray(unpack_genomes(packed, 32 * np.asarray(packed).shape[2])[:, order, :])


class ColumnBudget:
    """When the columns of a context run out (the host side of gnx_widen_cols).  A step adds at most per_step
    columns (MUT_MAX_NEW when non-neutral mutations can occur, else 0), so the columns in use are at most
    `bound`: the last count read plus per_step for every step enqueued since.  take(n, read_used) answers how
    many of n steps may be enqueued now and at which capacity; it calls read_used() (a synchronising read of
    the true count) only when the bound would pass the capacity, and then doubles the capacity until one
    more step fits (never past max_capacity, 128 * ceil(L / 128), which holds every locus)."""

    def __init__(self, used, capacity, per_step, max_capacity):
        self.bound, self.capacity = int(used), int(capacity)
        self.per_step, self.max_capacity = int(per_step), int(max_capacity)

    def take(self, n_steps, read_used):
        if self.capacity >= self.max_capacity or self.bound + self.per_step * n_steps <= self.capacity:
            self.bound += self.per_step * n_steps
            return n_steps, self.capacity
        self.bound = int(read_used())
        while self.bound + self.per_step > self.capacity and self.capacity < self.max_capacity:
            self.capacity = min(2 * self.capacity, self.max_capacity)
        k = n_steps if self.capacity >= self.max_capacity else min(n_steps, (self.capacity - self.bound) // self.per_step)
        self.bound += self.per_step * k
        return k, self.capacity
