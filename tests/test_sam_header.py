"""SAM output on the CPU: cbcg_sam_header on containers the CPU oracle writes (no device), its format errors, and the
restated MD rule (tests/sam_restate.py) against the synthetic generator's MD, which it writes canonically over an ACGT
genome."""
import numpy as np
import pytest

import oracle_lib as O
import sam_restate as R
from cbc_b200 import synth
from cbc_b200.codec import CbcgError, sam_header

ERR_FORMAT = -8


def _shape(seed, n_chr, lmin, lmax, p_indel, p_clip, n=4_000):
    cfg = synth.SynthConfig(seed=seed, genome_len=400_000, n_chr=n_chr, n_reads=n, len_min=lmin, len_max=lmax, p_sub=0.005,
                            p_indel=p_indel, p_clip=p_clip)
    g = synth.make_genome(cfg)
    return g, synth.make_reads(cfg, g)


def test_header_of_oracle_containers():
    for n_chr in (1, 3):
        g, b = _shape(5 + n_chr, n_chr, 100, 100, 0.002, 0.05)
        cont = O.encode_blocked(b, g, 100, 256)
        assert sam_header(cont) == R.header(g.names)


def test_malformed_headers():
    g, b = _shape(9, 2, 100, 100, 0.002, 0.05, n=500)
    cont = O.encode_blocked(b, g, 100, 128)
    bad_magic = b"XXXX" + cont[4:]
    bad_version = cont[:4] + (99).to_bytes(4, "little") + cont[8:]
    long_name = cont[:40] + (300).to_bytes(4, "little") + cont[44:]
    for data in (b"", cont[:39], bad_magic, bad_version, long_name, cont[:44]):
        with pytest.raises(CbcgError) as e:
            sam_header(data)
        assert e.value.status == ERR_FORMAT


@pytest.mark.parametrize("shape", ["config1", "config5"])
def test_md_rule_reproduces_the_generator(shape):
    if shape == "config1":
        g, b = _shape(71, 2, 100, 100, 0.002, 0.05)
    else:
        g, b = _shape(72, 2, 50, 250, 0.02, 0.3)
    up = R.upper(g)
    cig, seq, md = R.batch_cigars(b), R.batch_seqs(b), R.batch_mds(b)
    for i in range(b.n_reads):
        got, nm = R.md_nm(cig[i], seq[i], up[int(b.chr[i])], int(b.pos[i]))
        assert got == md[i], (i, cig[i])
        assert nm >= 0
    assert any(b"D" in c for c in cig) and any(b"S" in c for c in cig)
