"""Host mirror of the `cluster` subcommand: load one sketch file, and write its single-linkage ANI clusters
(hg_cluster_packed: unpack, dist windows and union-find all on the GPU; with a Group, hg_group_cluster_packed: one range
of the pairs per GPU, the forests united on GPU 0)."""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from . import fileio
from .dist import _stack_packed
from .ffi import Context, Group


@dataclass
class SketchCluster:
    path_sketch: str = ""
    out_file: str = ""
    ani_th: float = 95.0


def format_cluster_lines(names, rep) -> str:
    """One `rep_name\\tmember_name` line per sketch (galah's representative / member layout): clusters in ascending
    representative index, the representative's own line first, then the members in ascending index - the key
    (rep, t != rep, t).  A greedy representative (derep) need not be the smallest index of its cluster; a single-linkage
    one (cluster) always is, so there the key is (rep, t)."""
    rep = np.asarray(rep, np.int64)
    t = np.arange(rep.size)
    order = np.lexsort((t, t != rep, rep))
    return "".join("%s\t%s\n" % (names[rep[k]], names[k]) for k in order)


def cluster(sc: SketchCluster, ctx: Context | None = None, path: int = 0, group: Group | None = None) -> str:
    """Returns the text written to sc.out_file.  With `group` the run uses its GPUs (Group.cluster_packed)."""
    own = ctx is None and group is None
    if own:
        ctx = Context(0)
    try:
        sk = fileio.load_sketch(sc.path_sketch)
        if not sk:
            raise ValueError("empty sketch file")
        p, b, n = _stack_packed(sk)
        rep, _ = (group or ctx).cluster_packed(p, b, n, sk[0].hv_d, ksize=sk[0].ksize, ani_th=sc.ani_th, path=path)
        text = format_cluster_lines([s.file_str for s in sk], rep)
        if sc.out_file:
            with open(sc.out_file, "w") as f:
                f.write(text)
        return text
    finally:
        if own:
            ctx.close()
