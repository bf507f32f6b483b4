"""Host mirror of the `search` subcommand: load two sketch files, and for every query sketch write its top-k
best-matching refs (hg_search_packed: unpack, floor pass, main pass and selection all on the GPU; with a Group,
hg_group_search_packed: one block of refs per GPU, the blocks' results merged on GPU 0)."""
from __future__ import annotations

from dataclasses import dataclass

from . import fileio
from .dist import _stack_packed
from .ffi import Context, Group


@dataclass
class SketchSearch:
    path_ref_sketch: str = ""
    path_query_sketch: str = ""
    out_file: str = ""
    top_k: int = 10
    ani_min: float = 0.0


def format_search_lines(ref_names, qry_names, hits, n_found, milli) -> str:
    """One `ref\\tquery\\t{:.3}` line per result: queries in file order, each query's results in rank order."""
    out = []
    for j in range(len(qry_names)):
        for r in range(int(n_found[j])):
            m = int(milli[j, r])
            out.append("%s\t%s\t%d.%03d\n" % (ref_names[int(hits["i"][j, r])], qry_names[j], m // 1000, m % 1000))
    return "".join(out)


def search(ss: SketchSearch, ctx: Context | None = None, path: int = 0, group: Group | None = None) -> str:
    """Returns the text written to ss.out_file.  With `group` the search runs on its GPUs (Group.search_packed)."""
    own = ctx is None and group is None
    if own:
        ctx = Context(0)
    try:
        ref = fileio.load_sketch(ss.path_ref_sketch)
        qry = fileio.load_sketch(ss.path_query_sketch)
        if ref[0].ksize != qry[0].ksize:
            raise ValueError("Ref and query sketches use different kmer sizes!")  # dist.rs:29-32
        if ref[0].hv_d != qry[0].hv_d:
            raise ValueError("Ref and query sketches use different HV dimensions!")  # dist.rs:36-39
        hv_d, ksize = ref[0].hv_d, ref[0].ksize
        rp, rb, rn = _stack_packed(ref)
        qp, qb, qn = _stack_packed(qry)
        hits, n_found, milli = (group or ctx).search_packed(rp, rb, rn, qp, qb, qn, hv_d, ksize=ksize, top_k=ss.top_k,
                                                            ani_min=ss.ani_min, path=path)
        text = format_search_lines([s.file_str for s in ref], [s.file_str for s in qry], hits, n_found, milli)
        if ss.out_file:
            with open(ss.out_file, "w") as f:
                f.write(text)
        return text
    finally:
        if own:
            ctx.close()
