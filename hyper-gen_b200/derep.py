"""Host mirror of the `derep` subcommand: load one sketch file, and write its greedy ANI dereplication
(hg_derep_packed: unpack, the representatives' dist windows and greedy steps, and the assignment search all on the GPU)."""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from . import fileio
from .cluster import format_cluster_lines
from .dist import _stack_packed
from .ffi import Context

ORDERS = ("file", "size")


@dataclass
class SketchDerep:
    path_sketch: str = ""
    out_file: str = ""
    ani_th: float = 95.0
    order: str = "file"  # "file": file order; "size": descending hv_norm_2 (larger genomes first), ties by file index


def priority(norm2, order: str):
    """The priority order of the sketches: None for file order, else the permutation for `order`.  hv_norm_2 is about
    hv_d times the number of sampled hashes, so "size" puts the larger genomes first; it is the only priority a sketch
    file can give on its own."""
    if order not in ORDERS:
        raise ValueError("unknown order %r (expected one of %s)" % (order, ", ".join(ORDERS)))
    if order == "file":
        return None
    norm2 = np.asarray(norm2, np.int64)
    return np.lexsort((np.arange(norm2.size), -norm2)).astype(np.uint32)


def derep(sd: SketchDerep, ctx: Context | None = None, path: int = 0) -> str:
    """Returns the text written to sd.out_file: `rep\\tmember` lines as `cluster` writes them."""
    if sd.order not in ORDERS:  # before the file is read
        raise ValueError("unknown order %r (expected one of %s)" % (sd.order, ", ".join(ORDERS)))
    own = ctx is None
    if own:
        ctx = Context(0)
    try:
        sk = fileio.load_sketch(sd.path_sketch)
        if not sk:
            raise ValueError("empty sketch file")
        p, b, n = _stack_packed(sk)
        rep, _ = ctx.derep_packed(p, b, n, sk[0].hv_d, ksize=sk[0].ksize, ani_th=sd.ani_th, path=path, order=priority(n, sd.order))
        text = format_cluster_lines([s.file_str for s in sk], rep)
        if sd.out_file:
            with open(sd.out_file, "w") as f:
                f.write(text)
        return text
    finally:
        if own:
            ctx.close()
