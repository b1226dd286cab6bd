"""Phase order of one strip time step (geonomics_b200/strips.py `phase_sequence`, read from the
library's gnx_strip_phase_order, the table gnx_step runs; CPU): fixed births keep the eight phases
with the births all-gather after phase 3; Poisson births publish the pairs after phase 3, all-gather
them, and draw the births in phase 8 before the births all-gather."""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from geonomics_b200 import strips  # noqa: E402


def test_fixed_births_keep_the_eight_phases():
    seq = strips.phase_sequence(1)
    assert [k for k, _ in seq] == list(range(8))
    assert [s for _, s in seq] == [0, 0, 0, 1, 0, 2, 3, None]
    assert strips.phase_sequence(True) == seq


def test_poisson_births_gather_the_pairs_then_draw_in_phase_8():
    seq = strips.phase_sequence(0)
    assert seq == [(0, 0), (1, 0), (2, 0), (3, 4), (8, 1), (4, 0), (5, 2), (6, 3), (7, None)]
    assert strips.phase_sequence(False) == seq

