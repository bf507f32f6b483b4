"""Host side of the ANI matrix without a GPU: the PHYLIP lower-triangle text, the square it mirrors into, and the
entries in the ABI."""
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_triangle_text_is_phylip_lower_with_dist_rounding():
    from hypergen_b200.matrix import format_triangle
    # 97.0625 * 1000 = 97062.5 rounds to even; 99.99951 rounds up into the next integer
    tri = np.array([97.0625, 100.0, 0.0, 99.99951, 12.5, 85.1], np.float32)
    assert format_triangle(["a", "b", "c", "d"], tri) == (
        "4\na\nb\t97.062\nc\t100.000\t0.000\nd\t100.000\t12.500\t85.100\n")
    assert format_triangle([], np.zeros(0, np.float32)) == "0\n"
    assert format_triangle(["only"], np.zeros(0, np.float32)) == "1\nonly\n"
    with pytest.raises(ValueError, match="strict lower triangle"):
        format_triangle(["a", "b"], np.zeros(2, np.float32))


def test_square_mirrors_the_lower_triangle():
    from hypergen_b200.matrix import square_from_lower
    sq = square_from_lower(np.array([1, 2, 3], np.float32), 3)
    assert sq.tolist() == [[100, 1, 2], [1, 100, 3], [2, 3, 100]]
    assert square_from_lower(np.zeros(0, np.float32), 1, diagonal=0.0).tolist() == [[0.0]]


def test_matrix_entries_are_declared_and_bound():
    from hypergen_b200 import ffi
    src = open(os.path.join(ROOT, "include", "hypergen_b200.h")).read()
    names = ["hg_ani_matrix_dev", "hg_ani_matrix_packed", "hg_group_ani_matrix_packed", "hg_ani_matrix_stats"]
    for n in names:
        assert re.search(r"HG_API\s+int\s+%s\s*\(" % n, src), n
        assert n in ffi.EXPORTS, n
    rust = open(os.path.join(ROOT, "rust", "src", "hypergen_b200_sys.rs")).read()
    for n in names:
        assert "fn %s(" % n in rust, n


def test_a_caller_output_too_small_is_refused_before_the_call():
    from hypergen_b200 import ffi
    p = np.zeros((5, 512), np.uint8)
    b = np.full(5, 8, np.uint8)
    nm = np.ones(5, np.int32)
    q = (p[:3].copy(), b[:3].copy(), nm[:3].copy())

    def never(*args):
        raise AssertionError("the library was called")

    bad = [
        (True, np.empty(9, np.float32)),          # lower: 10 entries
        (True, np.empty((2, 5), np.float32)),     # lower: 1-D only
        (False, np.empty(14, np.float32)),        # 5 x 3
        (False, np.empty((4, 3), np.float32)),    # too few rows
        (False, np.empty((5, 2), np.float32)),    # rows too short
        (False, np.empty(15, np.float64)),
        (False, np.empty((5, 6), np.float32)[:, ::2]),
    ]
    for lower, out in bad:
        with pytest.raises(ValueError):
            ffi._ani_matrix_packed(never, None, p, b, nm, *((p, b, nm) if lower else q), 512, 21, 0, lower, out)
