"""The all-vs-all ANI matrix of a sketch file (hg_ani_matrix_packed: unpack, dense dist bands and the dot-to-ANI conversion
on the GPU), the square it mirrors into, and the Python mirror of `hyper-gen triangle`'s text."""
from __future__ import annotations

import numpy as np

from . import fileio
from .dist import _stack_packed
from .ffi import Context


def load_matrix(path_sketch: str, ctx: Context | None = None, lower: bool = True, path: int = 0):
    """(names, ani) of one sketch file: ani is the float32 strict lower triangle (n (n - 1) / 2 entries, row i holding
    j < i at i (i - 1) / 2 + j) or, with lower=False, the full n x n square (diagonal as the kernel gives it)."""
    own = ctx is None
    if own:
        ctx = Context(0)
    try:
        sk = fileio.load_sketch(path_sketch)
        if not sk:
            raise ValueError("empty sketch file")
        p, b, n = _stack_packed(sk)
        ani = ctx.ani_matrix_packed(p, b, n, hv_d=sk[0].hv_d, ksize=sk[0].ksize, path=path, lower=lower)
        return [s.file_str for s in sk], ani
    finally:
        if own:
            ctx.close()


def square_from_lower(tri, n: int, diagonal: float = 100.0) -> np.ndarray:
    """the symmetric n x n matrix of a strict lower triangle (PHYLIP order), `diagonal` on the diagonal"""
    tri = np.asarray(tri, np.float32)
    if tri.size != n * (n - 1) // 2:
        raise ValueError("a strict lower triangle of %d rows has %d entries, got %d" % (n, n * (n - 1) // 2, tri.size))
    out = np.full((n, n), np.float32(diagonal), np.float32)
    i, j = np.tril_indices(n, -1)
    out[i, j] = tri
    out[j, i] = tri
    return out


def format_triangle(names, tri) -> str:
    """`hyper-gen triangle`'s text: n, then per sketch its name and a tab plus ANI(i, j) for every j < i, each value as
    `dist` prints it (thousandths rounded half to even, printed as %u.%03u)."""
    n = len(names)
    tri = np.asarray(tri, np.float32)
    if tri.size != n * (n - 1) // 2:
        raise ValueError("a strict lower triangle of %d rows has %d entries, got %d" % (n, n * (n - 1) // 2, tri.size))
    milli = np.rint(tri.astype(np.float64) * 1000.0).astype(np.uint64)
    cells = ["%d.%03d" % (m // 1000, m % 1000) for m in milli.tolist()]
    lines = [str(n)]
    for i, name in enumerate(names):
        lines.append("\t".join([name] + cells[i * (i - 1) // 2: i * (i - 1) // 2 + i]))
    return "\n".join(lines) + "\n"


def triangle(path_sketch: str, out_file: str = "", ctx: Context | None = None, path: int = 0) -> str:
    """Returns the text `hyper-gen triangle -r path_sketch -o out_file` writes (and writes it when out_file is given)."""
    names, tri = load_matrix(path_sketch, ctx, lower=True, path=path)
    text = format_triangle(names, tri)
    if out_file:
        with open(out_file, "w") as f:
            f.write(text)
    return text
