"""Generates the golden fixtures in this directory from the UNMODIFIED reference (run in the build container,
where /root/reference exists and oracle/_ref has been built by `make -C oracle`):

  adversarial_input.npz          the packed adversarial batch (seed 7) — stored so the fixtures do not depend on
                                 numpy's generator staying bit-stable
  ref_<optionset>.npz            per-read records, pre/post Stats blocks and FilterResult counters produced by the
                                 reference's own operators (oracle/_ref/libfplref.so) for each tests/cases.py option set
  blocky_input.npz               the packed blocky-quality batch (seed 88) for the --mask/--break fixtures
  ref_mb_<set>.npz               the same for tests/cases.py MASK_BREAK_SETS, plus the output-read and masked-region lists
  binary_<name>.json             whole-binary runs of oracle/_ref/fastplong_ref on a seeded FASTQ: md5 of --out and
                                 --failed_out, md5 of the JSON report text minus its "command" line, the report's
                                 scalar sections (curves replaced by their md5), and the input md5
  reference_outputs.json         what the reference computed in the tests that compare with it (tests/reference_outputs.py):
                                 those tests are called here with the reference running in place of the stored outputs

Usage:  python tests/golden/make_golden.py [reference_outputs]     (the argument: only reference_outputs.json)
"""
import hashlib
import inspect
import itertools
import json
import os
import pathlib
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import cases  # noqa: E402
from fastplong_b200 import synth  # noqa: E402
from oracle_lib import REF_BIN, RefEngine  # noqa: E402

BINARY_RUNS = {
    # name: (seed, n_reads, mean_len, option set, extra synth kwargs)
    "c1_small": (11, 160, 1500, "default_se", {"p_chimera": 0.05, "q_mean": 17.0}),
    "cut_polyx": (12, 160, 1500, "cut_polyx_cplx", {"p_polya": 0.05, "p_chimera": 0.05, "q_mean": 17.0}),
    "loose": (13, 120, 1200, "loose_ed", {"p_chimera": 0.04}),
}
# --mask / --break whole-binary runs on cases.blocky_quality_batch(seed, n)
BINARY_MB_RUNS = {
    "mb_break": (21, 120, "break_default"),
    "mb_mask": (22, 120, "mask_cplx"),
    "mb_both": (23, 120, "mask_and_break"),
}


def md5(path):
    h = hashlib.md5()
    with open(path, "rb") as f:
        h.update(f.read())
    return h.hexdigest()


def json_digest(path):
    """md5 of the report text minus its "command" line (src/jsonreporter.cpp:91) + the scalar parts for reading."""
    lines = [ln for ln in open(path, "rb").read().split(b"\n") if b'"command"' not in ln]
    report = json.load(open(path))
    report.pop("command", None)
    for k in ("read_before_filtering", "read_after_filtering"):
        sec = report.get(k, {})
        for big in ("content_curves", "quality_curves", "kmer_count"):
            if big in sec:
                sec[big] = hashlib.md5(json.dumps(sec[big], sort_keys=True).encode()).hexdigest()
    return {"json_text_md5": hashlib.md5(b"\n".join(lines)).hexdigest(), "json": report}


def run_binary(binary, opt, fastq, outdir, threads=3):
    out, failed, js, html = (os.path.join(outdir, n) for n in ("out.fq", "failed.fq", "r.json", "r.html"))
    cmd = [binary, "-i", fastq, "-o", out, "--failed_out", failed, "-j", js, "-h", html, "-w", str(threads)]
    cmd += opt.cli_flags()
    subprocess.run(cmd, check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    return {"out_md5": md5(out), "failed_md5": md5(failed), **json_digest(js)}


def main():
    b = cases.adversarial_batch(7)
    np.savez_compressed(os.path.join(HERE, "adversarial_input.npz"), seq=b.seq, qual=b.qual, offsets=b.offsets,
                        lens=b.lens)
    cyc = int(b.lens.max())
    for name, opt in cases.OPTION_SETS.items():
        r = RefEngine(opt)
        res = r.process(b)
        np.savez_compressed(os.path.join(HERE, f"ref_{name}.npz"), results=res, pre=r.stats(0, cyc),
                            post=r.stats(1, cyc), counters=r.counters(), cycles=cyc)
    bb = cases.blocky_quality_batch(88, n=120)
    np.savez_compressed(os.path.join(HERE, "blocky_input.npz"), seq=bb.seq, qual=bb.qual, offsets=bb.offsets, lens=bb.lens)
    cyc = int(bb.lens.max())
    for name, opt in cases.MASK_BREAK_SETS.items():
        r = RefEngine(opt)
        res = r.process(bb)
        np.savez_compressed(os.path.join(HERE, f"ref_mb_{name}.npz"), results=res, pre=r.stats(0, cyc),
                            post=r.stats(1, cyc), counters=r.counters(), cycles=cyc, segments=r.segments(),
                            regions=r.mask_regions())
    for name, (seed, n, optname) in BINARY_MB_RUNS.items():
        opt = cases.MASK_BREAK_SETS[optname]
        batch = cases.blocky_quality_batch(seed, n=n)
        with tempfile.TemporaryDirectory() as d:
            fq = os.path.join(d, "in.fq")
            synth.to_fastq(batch, fq)
            g = run_binary(REF_BIN, opt, fq, d)
            g.update({"input_md5": md5(fq), "seed": seed, "n_reads": n, "options": optname})
        json.dump(g, open(os.path.join(HERE, f"binary_{name}.json"), "w"), indent=1, sort_keys=True)
    for name, (seed, n, mean, optname, kw) in BINARY_RUNS.items():
        opt = cases.OPTION_SETS[optname]
        batch = synth.ont_like(n, mean, seed, **kw)
        with tempfile.TemporaryDirectory() as d:
            fq = os.path.join(d, "in.fq")
            synth.to_fastq(batch, fq)
            g = run_binary(REF_BIN, opt, fq, d)
            g.update({"input_md5": md5(fq), "seed": seed, "n_reads": n, "mean_len": mean, "options": optname,
                      "synth_kwargs": kw})
        json.dump(g, open(os.path.join(HERE, f"binary_{name}.json"), "w"), indent=1, sort_keys=True)
    print("golden fixtures written to", HERE)


# the tests that compare with the reference; the GPU ones stop once the reference has run (reference_outputs.Recorded)
REFERENCE_TESTS = {
    "test_oracle_vs_reference": None,
    "test_evaluator": ["test_host_logic_matches_reference_binary"],
    "test_gpu_binary": ["test_gpu_binary_matches_reference_binary", "test_gpu_binary_mask_break_matches_reference_binary",
                        "test_config1_full_size_bit_exact", "test_gpu_binary_non_strict_fastq_like_reference",
                        "test_gpu_binary_many_small_chunks", "test_gpu_binary_file_size_is_a_multiple_of_the_chunk",
                        "test_gpu_binary_plus_lines_kept_verbatim"],
    "test_gpu_multigpu": ["test_drop_in_binary_workers_over_two_gpus"],
}


def parameter_sets(fn):
    """Every keyword set pytest would call `fn` with (its parametrize marks, crossed)."""
    axes = []
    for m in getattr(fn, "pytestmark", []):
        if m.name != "parametrize":
            continue
        names = [n.strip() for n in m.args[0].split(",")] if isinstance(m.args[0], str) else list(m.args[0])
        axes.append([dict(zip(names, v if len(names) > 1 else (v,))) for v in m.args[1]])
    for combo in itertools.product(*axes):
        yield {k: v for d in combo for k, v in d.items()}


def record_reference_outputs():
    import importlib
    import reference_outputs
    rec = reference_outputs.RECORDING = {}
    for modname, names in REFERENCE_TESTS.items():
        mod = importlib.import_module(modname)
        if modname == "test_gpu_multigpu":
            mod._n_gpus = lambda: 2              # only the reference half runs here
        reference_outputs.STOP_AFTER_RECORD = modname.startswith("test_gpu")
        for name in names or [n for n in dir(mod) if n.startswith("test_")]:
            fn = getattr(mod, name)
            for kw in parameter_sets(fn):
                keys = set(rec)
                with tempfile.TemporaryDirectory() as d:
                    if "tmp_path" in inspect.signature(fn).parameters:
                        kw["tmp_path"] = pathlib.Path(d)
                    try:
                        fn(**kw)
                    except reference_outputs.Recorded:
                        pass
                assert set(rec) != keys or modname.startswith("test_gpu"), (name, kw)
    reference_outputs.RECORDING = None
    with open(reference_outputs.PATH, "w") as f:
        json.dump(rec, f, indent=0, sort_keys=True)
        f.write("\n")
    print(len(rec), "reference outputs written to", reference_outputs.PATH)


if __name__ == "__main__":
    if sys.argv[1:] != ["reference_outputs"]:
        main()
    record_reference_outputs()
