"""Host side of `derep` without a GPU: the priority orders and the representative / member line layout."""
import numpy as np
import pytest


def test_size_order_is_descending_norm_then_file_index():
    from hypergen_b200 import derep
    assert derep.priority([5, 9, 9, 1], "file") is None
    assert derep.priority([5, 9, 9, 1], "size").tolist() == [1, 2, 0, 3]
    assert derep.priority(np.zeros(0, np.int32), "size").size == 0
    with pytest.raises(ValueError, match="unknown order"):
        derep.priority([1], "quality")


def test_lines_put_each_representative_first_even_above_its_members():
    from hypergen_b200.cluster import format_cluster_lines
    names = ["a", "b", "c", "d", "e"]
    # greedy labels: 2 represents 0, 1 and 4; 3 is its own
    assert format_cluster_lines(names, [2, 2, 2, 3, 2]) == "c\tc\nc\ta\nc\tb\nc\te\nd\td\n"
    # single-linkage labels (rep <= index) keep the order (rep, index)
    assert format_cluster_lines(names, [0, 0, 2, 0, 2]) == "a\ta\na\tb\na\td\nc\tc\nc\te\n"
