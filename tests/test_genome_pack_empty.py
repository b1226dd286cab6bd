"""genome_pack on zero individuals (CPU): a strip of a decomposed landscape may hold nobody, and its
share of a download is then an empty genome array."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from geonomics_b200 import genome_pack as gp  # noqa: E402


def test_unpack_of_no_individuals():
    assert gp.unpack_genomes(np.zeros((0, 2, 16), np.uint32), 512).shape == (0, 512, 2)
    assert gp.pack_genomes(np.zeros((0, 512, 2), np.int8)).shape[0] == 0
