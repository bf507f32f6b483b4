"""Host side of the FASTA records mode, without a GPU: the record naming rule of `hyper-gen sketch -i true` and its
Python mirror, and the layout of hg_fasta_record."""


def test_record_id_rule():
    from hypergen_b200 import sketch
    assert sketch.record_id("d/a.fna", b"NC_001.1 Escherichia coli", True, 3) == "NC_001.1"
    assert sketch.record_id("d/a.fna", b"contig7\tlen=500", True, 0) == "contig7"
    assert sketch.record_id("d/a.fna", b"plain", True, 0) == "plain"
    assert sketch.record_id("d/a.fna", b"", True, 2) == "d/a.fna#2"            # '>' alone
    assert sketch.record_id("d/a.fna", b" desc only", True, 1) == "d/a.fna#1"  # empty ID
    assert sketch.record_id("d/a.fna", b"", False, 0) == "d/a.fna#0"           # sequence before the first header


def test_record_struct_layout(hg):
    assert hg.ffi.RECORD_DTYPE.itemsize == 32
    assert [hg.ffi.RECORD_DTYPE.fields[k][1] for k in ("name_off", "name_len", "seq_len", "file", "has_header")] == [0, 8, 16, 24, 28]
