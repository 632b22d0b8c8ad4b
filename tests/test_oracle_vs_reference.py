"""Differential test: the oracle restatement vs the UNMODIFIED reference operators on seeded batches beyond the committed
fixtures.  The reference's outputs (oracle/_ref/libfplref.so, run by tests/golden/make_golden.py on these same inputs) are
stored as digests in tests/golden/reference_outputs.json (tests/reference_outputs.py)."""
import numpy as np
import pytest

import cases
from fastplong_b200 import Options, pack_reads, synth
from oracle_lib import OracleEngine, RefEngine
from reference_outputs import digest, expected


def outputs(eng, batch, lists=False):
    """Digests of everything one engine computes on a batch: records, both Stats blocks, counters and, under --mask /
    --break, the output-read and masked-region lists."""
    out = {"input": digest(np.concatenate([batch.seq, batch.qual, batch.offsets.view(np.uint8), batch.lens.view(np.uint8)])),
           "results": digest(eng.process(batch))}
    if lists:
        out["segments"] = digest(eng.segments())
        out["regions"] = digest(eng.mask_regions())
    cyc = max(1, int(batch.lens.max()) if batch.n_reads else 1)
    for w in (0, 1):
        out[f"stats{w}"] = digest(eng.stats(w, cyc))
    out["counters"] = digest(eng.counters())
    return out


def check(opt, batch, key, lists=False, note=""):
    ref = expected(key, lambda: outputs(RefEngine(opt), batch, lists))
    got = outputs(OracleEngine(opt), batch, lists)
    assert got["input"] == ref["input"], f"{key}: the seeded input is not the one the reference ran on {note}"
    for part in ref:
        assert got[part] == ref[part], f"{key}: oracle {part} differs from the reference's {note}"


@pytest.mark.parametrize("name", sorted(cases.OPTION_SETS))
@pytest.mark.parametrize("seed", [1, 2])
def test_adversarial(name, seed):
    check(cases.OPTION_SETS[name], cases.adversarial_batch(seed), f"{name}/adv{seed}")


@pytest.mark.parametrize("name", sorted(cases.OPTION_SETS))
def test_ont_like(name):
    check(cases.OPTION_SETS[name], cases.ont_batch(77, n=150, mean=2500, p_chimera=0.05, p_polya=0.05), name + "/ont")


@pytest.mark.parametrize("n", sorted(cases.LONG_ADAPTERS))
def test_long_adapters(n):
    check(cases.OPTION_SETS[f"long_adapter_{n}"], cases.long_adapter_batch(n, 900 + n), f"long{n}")


def test_edit_distance_random_pairs():
    rng = np.random.default_rng(5)
    pairs = []
    for _ in range(3000):
        la, lb = int(rng.integers(0, 150)), int(rng.integers(0, 150))
        a = synth.BASES[rng.integers(0, 4, size=la)].tobytes()
        b = synth.BASES[rng.integers(0, 4, size=lb)].tobytes()
        if rng.random() < 0.5 and la:
            b = a[: int(rng.integers(0, la + 1))] + b[: int(rng.integers(0, 6))]
        pairs.append((a, b))
    for la, lb in ((700, 650), (641, 10), (64, 65), (128, 129), (640, 640)):
        pairs.append((synth.BASES[rng.integers(0, 4, size=la)].tobytes(), synth.BASES[rng.integers(0, 4, size=lb)].tobytes()))
    distances = lambda eng: [eng.edit_distance(a, b) for a, b in pairs]
    inp = digest(np.frombuffer(b"|".join(a + b"," + b for a, b in pairs), np.uint8))
    ref = expected("edit_distance_random_pairs", lambda: {"input": inp, "distances": distances(RefEngine(Options()))})
    assert inp == ref["input"], "the seeded pairs are not the ones the reference ran on"
    got = distances(OracleEngine(Options()))
    for i, (d, r) in enumerate(zip(got, ref["distances"])):
        assert d == r, (i, len(pairs[i][0]), len(pairs[i][1]), d, r)
    assert len(got) == len(ref["distances"])


@pytest.mark.parametrize("name", sorted(cases.RNA_SETS))
@pytest.mark.parametrize("mixed", [False, True])
def test_rna_reads(name, mixed):
    """U instead of T: 5-mers through base2val's U case, content bin 5, byte-wise adapter comparison, polyX that does not
    count U."""
    batch = cases.rna_batch(41, mixed=mixed)
    assert (batch.seq == ord("U")).sum() > 10000
    check(cases.RNA_SETS[name], batch, f"{name}/rna{int(mixed)}")


@pytest.mark.parametrize("name", sorted(cases.edge_cases()))
def test_crafted_boundary_cases(name):
    """cases.edge_cases(): the boundaries a mutation run over the oracle found unpinned (more events than inline slots, global
    trims that eat the read exactly, a cut from one side with a trim on the other, N inside polyX runs, one filter without
    the other, ties of the filter thresholds)."""
    opt, batch = cases.edge_cases()[name]
    check(opt, batch, "edge/" + name)


@pytest.mark.parametrize("name", sorted(cases.EXTREME_SETS))
def test_extreme_option_values(name):
    opt = cases.EXTREME_SETS[name]
    batch = cases.ont_batch(8, n=40, mean=2500, p_chimera=0.2, p_polya=0.2) if name == "fasta_200_entries" else cases.adversarial_batch(12)
    check(opt, batch, "extreme/" + name, lists=bool(opt.mask or opt.break_reads))


def test_empty_batch():
    check(cases.OPTION_SETS["default_se"], pack_reads([]), "empty")


@pytest.mark.parametrize("name", sorted(cases.MASK_BREAK_SETS))
@pytest.mark.parametrize("kind", ["blocky", "adversarial", "ont"])
def test_mask_break(name, kind):
    """--mask / --break: records, the output-read list, the masked regions, both Stats blocks, counters."""
    opt = cases.MASK_BREAK_SETS[name]
    batch = {"blocky": lambda: cases.blocky_quality_batch(5, n=100), "adversarial": lambda: cases.adversarial_batch(4),
             "ont": lambda: cases.ont_batch(6, n=80, mean=2000, p_chimera=0.05)}[kind]()
    check(opt, batch, f"{name}/{kind}", lists=True)


@pytest.mark.parametrize("seed", [31, 32, 33])
def test_random_option_sets(seed):
    """Seeded random option sets x batches (cases.random_case; tools/fuzz_oracle_vs_reference.py runs the same for longer)."""
    import random
    rng = random.Random(seed)
    for i in range(40):
        opt, batch, what = cases.random_case(rng)
        check(opt, batch, f"random{seed}/{i}", lists=bool(opt.mask or opt.break_reads), note=what)
