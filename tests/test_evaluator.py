"""Adapter auto-detection (SURVEY §8f row 4): fastplong_b200/evaluator.py (host half) against the unmodified reference
binary's own detection, and the device ten-mer tables against their numpy restatement."""
import json
import subprocess

import numpy as np
import pytest

from fastplong_b200 import evaluator, synth
from oracle_lib import REF_BIN, kmer10_tables
from reference_outputs import digest, expected


def reference_detection(batch, tmp_path, extra=()):
    fq = str(tmp_path / "in.fq")
    synth.to_fastq(batch, fq)
    js = str(tmp_path / "ref.json")
    r = subprocess.run([REF_BIN, "-i", fq, "-o", str(tmp_path / "o.fq"), "-j", js, "-h", str(tmp_path / "r.html"), "-w", "2", *extra],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-1000:]
    j = json.load(open(js))
    ac = j.get("adapter_cutting", {})
    return ac.get("read_start_adapter"), ac.get("read_end_adapter"), r.stderr


@pytest.mark.parametrize("seed,kw", [(5, {}), (6, dict(p_start=0.5, p_end=0.9)), (7, dict(p_start=0.05, p_end=0.6)),
                                     (8, dict(adapter_start="GATCGGAAGAGCACACGTCTGAACTCCAGTCAC", adapter_end="ACACTCTTTCCCTACACGACGCTCTTCCGATCT"))])
def test_host_logic_matches_reference_binary(seed, kw, tmp_path):
    """The adapters the reference binary detected on these seeded reads (stored, tests/reference_outputs.py)."""
    batch = synth.ont_like(600, 1500, seed, **kw)
    inp = digest(np.concatenate([batch.seq, batch.qual]))
    def run_reference():
        start, end, _ = reference_detection(batch, tmp_path)
        return {"input": inp, "start": start, "end": end}
    ref = expected(f"evaluator/{seed}", run_reference)
    assert ref["input"] == inp, "the seeded reads are not the ones the reference ran on"
    start, end = ref["start"], ref["end"]
    # the JSON prints "unspecified" for an adapter left at "auto" (src/options.cpp:247-259)
    norm = lambda s: "unspecified" if s == "auto" else s
    for pick in ("abi", "python"):       # the C ABI's fpl_eval_pick_adapter and its Python twin
        got = evaluator.detect_adapters(batch, kmers=kmer10_tables, pick=pick)
        assert (norm(got[0]), norm(got[1])) == (start, end), pick


def _planted_tables(rng):
    """Ten-mer tables with a chain of overlapping ten-mers of one random sequence planted at decaying counts over sparse
    noise: the regime where the extension rules (70 % of the neighbours, half of the key's count, offset window) decide."""
    counts = np.zeros(1 << 20, dtype=np.uint32)
    acc = np.zeros(1 << 20, dtype=np.uint64)
    noise = rng.integers(0, 1 << 20, size=int(rng.integers(20000, 80000)))     # mostly singletons, like random read ends
    np.add.at(counts, noise, 1)
    acc[:] = counts.astype(np.uint64) * np.uint64(rng.integers(0, 120))
    kind = rng.integers(0, 4)
    n = int(rng.integers(14, 80))
    if kind == 0:
        seq = rng.integers(0, 4, size=n)
    elif kind == 1:                       # runs of A: neighbours of the planted keys include AAAAAAAAAA (its count is ignored)
        seq = np.where(rng.random(n) < 0.6, 0, rng.integers(0, 4, size=n))
    elif kind == 2:                       # short period
        seq = np.resize(rng.integers(0, 4, size=int(rng.integers(2, 7))), n)
    else:                                 # C/G rich
        seq = rng.choice([2, 3, 2, 3, 0, 1], size=n)
    base = int(rng.integers(11, 900))
    start = int(rng.integers(0, 60))
    for i in range(n - 9):
        key = 0
        for b in seq[i:i + 10]:
            key = (key << 2) | int(b)
        c = max(0, int(base * rng.uniform(*[(0.75, 1.1), (0.75, 1.1), (0.4, 1.2)][int(rng.integers(3))])))
        counts[key] += c
        acc[key] += np.uint64(max(0, c * (start + i) + int(rng.integers(-c, c + 1) * rng.choice([0.3, 0.3, 2.5]))))
    total = int(counts.sum() * rng.choice([1, 1, 1, 30]))
    return counts, acc, total


def test_abi_pick_equals_python_twin_on_planted_tables():
    """fpl_eval_pick_adapter (C++, include/fplgpu.h) against evaluator.detect_one on 40 synthetic table pairs, DNA and RNA;
    neither modifies its input."""
    from fastplong_b200.binding import eval_pick_adapter
    rng = np.random.default_rng(2026)
    found = 0
    for case in range(40):
        counts, acc, total = _planted_tables(rng)
        c0, a0 = counts.copy(), acc.copy()
        for rna in (False, True):
            got = eval_pick_adapter(counts, acc, total, rna)
            exp = evaluator.detect_one(counts, acc, total, rna)
            assert got == exp, (case, rna, got, exp)
            found += got is not None
        assert np.array_equal(counts, c0) and np.array_equal(acc, a0)
    assert found > 10


def test_abi_pick_rejects_bad_arguments():
    from fastplong_b200 import binding
    lib = binding.load_library()
    c = np.zeros(1 << 20, dtype=np.uint32)
    a = np.zeros(1 << 20, dtype=np.uint64)
    import ctypes as C
    buf = C.create_string_buffer(80)
    assert lib.fpl_eval_pick_adapter(c.ctypes.data, a.ctypes.data, 0, 0, buf, 80) == 0 and buf.value == b""
    assert lib.fpl_eval_pick_adapter(c.ctypes.data, a.ctypes.data, 0, 0, buf, 64) < 0
    assert lib.fpl_eval_pick_adapter(None, a.ctypes.data, 0, 0, buf, 80) < 0
    with pytest.raises(binding.FplError):
        binding.eval_pick_adapter(c[:100], a, 0)


def test_fewer_than_100_reads_detects_nothing():
    batch = synth.ont_like(60, 800, 3)
    assert evaluator.detect_adapters(batch, kmers=kmer10_tables) == ("auto", "auto")


def test_evaluated_prefix_limits():
    assert evaluator.evaluated_prefix([10] * 5) == 5
    assert evaluator.evaluated_prefix([1000] * 70000) == 64 * 1024
    lens = [300_000_000, 300_000_000, 5, 5]
    assert evaluator.evaluated_prefix(lens) == 2          # the read that crosses 512 Mi bases is still loaded


@pytest.mark.gpu
@pytest.mark.parametrize("side", [0, 1])
def test_device_tables_match_numpy(side):
    from fastplong_b200.binding import eval_adapter_kmers
    from fastplong_b200 import pack_reads
    reads = synth.adversarial_reads(9) + [synth.ont_like(300, 900, 4).read(i) for i in range(300)]
    batch = pack_reads(reads)
    for shift in (1, 3):
        c, a, t = eval_adapter_kmers(batch, side, shift)
        rc, ra, rt = kmer10_tables(batch, side, shift)
        assert t == rt and np.array_equal(c, rc) and np.array_equal(a, ra)


@pytest.mark.gpu
def test_device_detection_finds_the_planted_adapters():
    batch = synth.ont_like(800, 2000, 21)
    assert evaluator.detect_adapters(batch) == (synth.ADAPTER_START, synth.ADAPTER_END)


def test_reference_known_answer_int2seq_roundtrip():
    """The reference's own evaluator test (test/evaluator_test.cpp:4-8): int2seq(seq2int("ATCGATCGAT")) is the string —
    here with the ten-mer table as seq2int (the only key counted for that read is the string's) and both int2seq forms."""
    from fastplong_b200 import pack_reads
    s = b"ATCGATCGAT"
    batch = pack_reads([(s + b"A", b"I" * 11)])           # shift_tail 1: exactly one ten-mer position
    counts, acc, total = kmer10_tables(batch, 0, 1)
    keys = np.nonzero(counts)[0]
    assert total == 1 and len(keys) == 1
    assert evaluator.int2seq(int(keys[0])) == s.decode()
    assert evaluator.int2seq(int(keys[0]), is_rna=True) == s.decode().replace("T", "U")
