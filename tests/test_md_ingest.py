"""Host C ingest of SAM without MD tags (CBCH_DERIVE_MD, cbch_read_sam_ex) and the compact packing of a batch without MD
(cbch_pack_batch): the batch the library derives MD for on the GPU. CPU only."""
import ctypes as C
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

from cbc_b200 import synth
from cbc_b200.codec import CompactBatch
from test_host_ingest import Fasta, HBatch, LIB, ROOT, _arr

CBCH_DERIVE_MD = 1
CFG = dict(seed=34, genome_len=300_000, n_chr=3, n_reads=6000, len_min=50, len_max=250, p_sub=0.01, p_indel=0.02, p_clip=0.3)


@pytest.fixture(scope="module")
def lib():
    subprocess.run(["make", "-s", "-C", ROOT, "host"], check=True)
    l = C.CDLL(LIB)
    l.cbch_read_fasta.argtypes = [C.c_char_p, C.POINTER(Fasta), C.c_char_p, C.c_size_t]
    l.cbch_read_sam.argtypes = [C.c_char_p, C.POINTER(Fasta), C.c_int, C.POINTER(HBatch), C.c_char_p, C.c_size_t]
    l.cbch_read_sam_ex.argtypes = [C.c_char_p, C.POINTER(Fasta), C.c_int, C.c_int, C.c_uint32, C.POINTER(HBatch), C.c_char_p, C.c_size_t]
    return l


def _strip_md(text: str) -> str:
    return re.sub(r"\tMD:Z:[^\t\n]*", "", text)


@pytest.fixture(scope="module")
def files():
    cfg = synth.SynthConfig(**CFG)
    g = synth.make_genome(cfg); b = synth.make_reads(cfg, g)
    with tempfile.TemporaryDirectory() as d:
        fa, sam, bare = (os.path.join(d, x) for x in ("r.fa", "r.sam", "bare.sam"))
        synth.write_fasta(fa, g); synth.write_sam(sam, b, g)
        with open(sam) as f:
            text = f.read()
        assert "\tMD:Z:" in text
        with open(bare, "w") as f:
            f.write(_strip_md(text))
        yield g, b, fa, sam, bare


def _read(lib, sam, fa, flags, threads=4):
    f, hb = Fasta(), HBatch()
    err = C.create_string_buffer(256)
    assert lib.cbch_read_fasta(fa.encode(), C.byref(f), err, 256) == 0, err.value
    rc = lib.cbch_read_sam_ex(sam.encode(), C.byref(f), 1, threads, flags, C.byref(hb), err, 256)
    return rc, hb, err.value.decode()


def _check_no_md(hb, b):
    n = hb.n_reads
    assert n == b.n_reads
    assert not hb.md_off and not hb.md                           # NULL pointers
    assert np.array_equal(_arr(hb.pos, n, np.uint32), b.pos) and np.array_equal(_arr(hb.flag, n, np.uint16), b.flag)
    assert np.array_equal(_arr(hb.seq_len, n, np.uint16), b.seq_len) and np.array_equal(_arr(hb.chr, n, np.uint32), b.chr)
    for name in ("seq", "cigar"):
        off = _arr(getattr(hb, name + "_off"), n + 1, np.uint64)
        assert np.array_equal(off, getattr(b, name + "_off"))
        assert np.array_equal(_arr(getattr(hb, name), int(off[-1]), np.uint8), getattr(b, name)[:int(off[-1])])
    assert hb.read_len_header == int(b.seq_len.max()) and hb.max_len == int(b.seq_len.max())


@pytest.mark.parametrize("threads", [1, 7])
def test_stripped_file_parses_to_the_batch_without_md(lib, files, threads):
    g, b, fa, sam, bare = files
    rc, hb, err = _read(lib, bare, fa, CBCH_DERIVE_MD, threads)
    assert rc == 0, err
    _check_no_md(hb, b)


def test_md_tags_that_are_present_are_ignored(lib, files):
    g, b, fa, sam, bare = files
    rc, hb, err = _read(lib, sam, fa, CBCH_DERIVE_MD)
    assert rc == 0, err
    _check_no_md(hb, b)


def test_without_the_flag_a_record_without_md_is_still_an_error(lib, files):
    g, b, fa, sam, bare = files
    rc, _, err = _read(lib, bare, fa, 0)
    assert rc == -5 and "MD" in err
    f, hb = Fasta(), HBatch()
    e = C.create_string_buffer(256)
    assert lib.cbch_read_fasta(fa.encode(), C.byref(f), e, 256) == 0
    assert lib.cbch_read_sam(bare.encode(), C.byref(f), 1, C.byref(hb), e, 256) == -5


def test_pack_batch_without_md(files):
    """A batch without MD packs to NULL md_len / md and a zero MD column; every other field as the batch with MD packs."""
    g, b, fa, sam, bare = files

    def arr(ptr, ct, m):
        return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(ct)), (m,)).copy() if m else np.zeros(0, np.uint8)
    full, bare_c = CompactBatch(b, pinned=False, threads=3), CompactBatch(b.without_md(), pinned=False, threads=3)
    v, w = full.c.v, bare_c.c.v
    n = b.n_reads
    assert not w.md_len and not w.md
    tiles = (n + 127) // 128 + 1
    tv = arr(v.tile_base, C.c_uint64, 4 * tiles).reshape(-1, 4)
    tw = arr(w.tile_base, C.c_uint64, 4 * tiles).reshape(-1, 4)
    assert not tw[:, 3].any() and np.array_equal(tv[:, :3], tw[:, :3])
    for name in ("n_reads", "n_runs", "n_exc", "max_len", "min_len"):
        assert getattr(v, name) == getattr(w, name), name
    nb = int(((b.seq_len.astype(np.int64) + 3) // 4).sum())
    for name, ct, m in (("pos", C.c_uint32, n), ("flag", C.c_uint16, n), ("seq_len", C.c_uint16, n), ("cigar_len", C.c_uint16, n),
                        ("run_first", C.c_uint64, v.n_runs), ("run_chr", C.c_uint32, v.n_runs), ("seq2", C.c_uint8, nb),
                        ("exc_read", C.c_uint32, v.n_exc), ("exc_base", C.c_uint16, v.n_exc), ("exc_char", C.c_uint8, v.n_exc),
                        ("cigar", C.c_uint8, int(b.cigar_off[n]))):
        assert np.array_equal(arr(getattr(v, name), ct, m), arr(getattr(w, name), ct, m)), name
    assert full.link_bytes - bare_c.link_bytes == 2 * n + int(b.md_off[n])
    full.close(); bare_c.close()
