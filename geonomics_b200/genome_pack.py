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
