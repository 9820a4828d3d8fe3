"""The edge-read catalogue (tests/edge_reads.py) through the CPU oracle: every case keeps the property it exists for,
extraction and reconstruction give the input back, coded cases round-trip through the single stream and blocked
containers, and refused cases are refused. Among them is a 20-base read with 255 deletions, whose edits outgrow any
bound proportional to the read's length."""
import numpy as np
import pytest

import edge_reads as E
import oracle_lib as O

_, GENOME = E.make_genomes()
CASES = E.cases(GENOME)
BLOCKED = [(1, 0), (16, 0), (16, 1), (1000, 1)]       # (block_reads, gen_mode)


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_extract_and_reconstruct(case):
    b = case.batch
    if not case.extract_ok:
        with pytest.raises(RuntimeError, match="cbco_extract"):
            O.extract(b, GENOME)
        return
    recs, edits = O.extract(b, GENOME)
    if case.check:
        case.check(b, recs, edits)
    assert O.reconstruct(recs, edits, b.chr, GENOME) == b.seq_lines()


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_single_stream(case):
    b = case.batch
    if not case.legacy_ok:
        with pytest.raises(RuntimeError, match="cbco_"):
            O.encode_legacy(b, GENOME, case.L)
        return
    stream, _ = O.encode_legacy(b, GENOME, case.L)
    assert O.decode_legacy(stream, GENOME) == (b.seq_lines(), b.n_reads)


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_blocked_container(case):
    b = case.batch
    for block_reads, gen_mode in BLOCKED:
        if not case.blocked_ok:
            with pytest.raises(RuntimeError, match="cbco_"):
                O.encode_blocked(b, GENOME, case.L, block_reads, gen_mode)
            continue
        cont = O.encode_blocked(b, GENOME, case.L, block_reads, gen_mode)
        assert O.decode_blocked(cont, GENOME) == (b.seq_lines(), b.n_reads), (block_reads, gen_mode)


def test_every_kind_of_refusal_is_in_the_catalogue():
    refused = {c.name for c in CASES if not c.extract_ok}
    assert {"del_run_256_refused", "one_past_chr_end_refused", "deletion_past_chr_end_refused"} <= refused
    alphabet = {c.name for c in CASES if c.extract_ok and not c.legacy_ok and not c.blocked_ok}
    assert {"snps_L_refused", "del_run_255_refused"} <= alphabet
    steps = {c.name for c in CASES if c.extract_ok and not c.legacy_ok and c.blocked_ok}
    assert {f"pos_step_{E.MAX_POS_X + 1}", "pos_step_6000000", "pos_step_11000000", "pos_steps_in_one_block"} <= steps


def test_the_255_deletion_read_is_extracted_in_full():
    """10M255D10M: 20 bases, 255 deletion entries. The oracle used to size its edit buffer by the read's length."""
    b = next(c for c in CASES if c.name == "del_run_255_refused").batch
    recs, edits = O.extract(b, GENOME)
    assert int(recs["n_dels"][-1]) == 255 and len(edits) >= 255
    assert O.reconstruct(recs, edits, b.chr, GENOME) == b.seq_lines()
