"""Whole-binary parity: build/fastplong_gpu (the reference CLI with our SingleEndProcessor + libfplgpu.so) against
what oracle/_ref/fastplong_ref (the unmodified reference) wrote for the same seeded inputs (stored,
tests/reference_outputs.py) and against the committed golden runs: md5 of --out and --failed_out, and the JSON report
text minus its "command" line (SURVEY §8c)."""
import hashlib
import json
import os
import subprocess

import pytest

import cases
from fastplong_b200 import synth
from oracle_lib import REF_BIN
from reference_outputs import expected

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GPU_BIN = os.environ.get("FPL_GPU_BIN") or os.path.join(ROOT, "build", "fastplong_gpu")      # FPL_EMULATE=1 (conftest.py) points this at the emulated build
GOLDEN = os.path.join(ROOT, "tests", "golden")


PARSE_ENV = {"device": None, "host": {"FPL_HOST_PARSE": "1"}, "device+emit": {"FPL_DEVICE_EMIT": "1"}}


def md5(path):
    return hashlib.md5(open(path, "rb").read()).hexdigest()


def json_text_md5(path):
    lines = [ln for ln in open(path, "rb").read().split(b"\n") if b'"command"' not in ln]
    return hashlib.md5(b"\n".join(lines)).hexdigest()


def run(binary, opt, fq, outdir, tag, threads=3, extra=(), env=None):
    out, failed, js, html = (os.path.join(outdir, f"{tag}.{n}") for n in ("out.fq", "failed.fq", "json", "html"))
    cmd = [binary, "-i", fq, "-o", out, "--failed_out", failed, "-j", js, "-h", html, "-w", str(threads)]
    cmd += opt.cli_flags() + list(extra)
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ, **(env or {})))
    assert r.returncode == 0, r.stderr[-2000:]
    return {"out_md5": md5(out), "failed_md5": md5(failed), "json_text_md5": json_text_md5(js), "json": js}


def reference_run(key, opt, fq, outdir, threads, extra=()):
    """The md5s of what the reference binary wrote for this input and these options."""
    inp = md5(fq)
    ref = expected("binary/" + key, lambda: dict(run(REF_BIN, opt, fq, outdir, "ref", threads, extra), json=None, input_md5=inp))
    assert ref["input_md5"] == inp, f"{key}: the seeded input is not the one the reference ran on"
    return ref


needs_bin = pytest.mark.skipif(not os.path.exists(GPU_BIN), reason="build/fastplong_gpu not built")


@needs_bin
@pytest.mark.parametrize("name", ["c1_small", "cut_polyx", "loose"])
def test_gpu_binary_matches_golden_reference_run(name, tmp_path):
    g = json.load(open(os.path.join(GOLDEN, f"binary_{name}.json")))
    batch = synth.ont_like(g["n_reads"], g["mean_len"], g["seed"], **g["synth_kwargs"])
    fq = str(tmp_path / "in.fq")
    synth.to_fastq(batch, fq)
    if md5(fq) != g["input_md5"]:
        pytest.skip("synthetic input differs from the fixture's")
    got = run(GPU_BIN, cases.OPTION_SETS[g["options"]], fq, str(tmp_path), "gpu")
    assert got["out_md5"] == g["out_md5"]
    assert got["failed_md5"] == g["failed_md5"]
    assert got["json_text_md5"] == g["json_text_md5"]


@needs_bin
@pytest.mark.parametrize("parse", ["device", "host", "device+emit"])
@pytest.mark.parametrize("name,threads", [("default_se", 1), ("cut_polyx_cplx", 4), ("fasta5", 3), ("literal_auto", 2),
                                          ("trims_limits", 3), ("end_only_wide_window", 8), ("fasta64_polyx", 5)])
def test_gpu_binary_matches_reference_binary(name, threads, parse, tmp_path):
    """Fresh input, both binaries side by side (config-1 shape: ONT-like reads, known 30 bp adapters), with the FASTQ
    parsed on the device (default for plain files), by the reference's FastqReader (FPL_HOST_PARSE=1), and parsed on the
    device with the output text assembled there too (FPL_DEVICE_EMIT=1, fpl_emit_fastq_host)."""
    opt = cases.OPTION_SETS[name]
    batch = synth.ont_like(700, 4000, 31 + threads, p_chimera=0.03, p_polya=0.03, q_mean=17.0)
    fq = str(tmp_path / "in.fq")
    synth.to_fastq(batch, fq)
    extra = []
    if opt.adapter_fasta:
        fa = str(tmp_path / "adapters.fa")
        with open(fa, "w") as f:   # headers chosen so that std::map order == list order (src/options.cpp:50-59)
            for i, s in enumerate(opt.adapter_fasta):
                f.write(f">a{i:03d}\n{s}\n")
        extra = ["-a", fa]
    ref = reference_run(f"{name}/w{threads}", opt, fq, str(tmp_path), threads, extra)
    got = run(GPU_BIN, opt, fq, str(tmp_path), "gpu", threads, extra, env=PARSE_ENV[parse])
    assert got["out_md5"] == ref["out_md5"]
    assert got["failed_md5"] == ref["failed_md5"]
    assert got["json_text_md5"] == ref["json_text_md5"]


@needs_bin
@pytest.mark.parametrize("name", ["mb_break", "mb_mask", "mb_both"])
def test_gpu_binary_mask_break_matches_golden_reference_run(name, tmp_path):
    g = json.load(open(os.path.join(GOLDEN, f"binary_{name}.json")))
    batch = cases.blocky_quality_batch(g["seed"], n=g["n_reads"])
    fq = str(tmp_path / "in.fq")
    synth.to_fastq(batch, fq)
    if md5(fq) != g["input_md5"]:
        pytest.skip("synthetic input differs from the fixture's")
    got = run(GPU_BIN, cases.MASK_BREAK_SETS[g["options"]], fq, str(tmp_path), "gpu")
    assert got["out_md5"] == g["out_md5"]
    assert got["failed_md5"] == g["failed_md5"]
    assert got["json_text_md5"] == g["json_text_md5"]


@needs_bin
@pytest.mark.parametrize("parse", ["device", "host", "device+emit"])
@pytest.mark.parametrize("name,threads", [("break_default", 2), ("break_w20", 3), ("mask_default", 1), ("mask_cplx", 4),
                                          ("mask_and_break", 3), ("break_no_adapter", 2)])
def test_gpu_binary_mask_break_matches_reference_binary(name, threads, parse, tmp_path):
    """-N / -b (SURVEY §8f row 3): both binaries side by side on blocky-quality reads, both parse paths."""
    opt = cases.MASK_BREAK_SETS[name]
    batch = cases.blocky_quality_batch(40 + threads, n=400)
    fq = str(tmp_path / "in.fq")
    synth.to_fastq(batch, fq)
    ref = reference_run(f"mb/{name}/w{threads}", opt, fq, str(tmp_path), threads)
    got = run(GPU_BIN, opt, fq, str(tmp_path), "gpu", threads, env=PARSE_ENV[parse])
    assert got["out_md5"] == ref["out_md5"]
    assert got["failed_md5"] == ref["failed_md5"]
    assert got["json_text_md5"] == ref["json_text_md5"]


@needs_bin
def test_config1_full_size_bit_exact(tmp_path):
    """BASELINE configs[0] at full size: 10k ONT reads mean 8 kb, known 30 bp start/end adapters, default Q-filter —
    the reference CPU run's outputs vs the GPU binary, bit-exact FASTQ outputs and JSON report; prints the GPU wall times."""
    import time
    opt = cases.OPTION_SETS["default_se"]
    batch = synth.ont_like(10000, 8000, 1)
    fq = "/dev/shm/fpl_c1_%d.fq" % os.getpid() if os.path.isdir("/dev/shm") else str(tmp_path / "c1.fq")
    synth.to_fastq(batch, fq)
    try:
        ref = reference_run("config1", opt, fq, str(tmp_path), 16)
        t1 = time.perf_counter()
        got = run(GPU_BIN, opt, fq, str(tmp_path), "gpu", threads=4)
        t2 = time.perf_counter()
        got_host = run(GPU_BIN, opt, fq, str(tmp_path), "gpuh", threads=4, env={"FPL_HOST_PARSE": "1"})
        t3 = time.perf_counter()
    finally:
        if fq.startswith("/dev/shm"):
            os.remove(fq)
    print(f"\nconfig 1 ({batch.n_bases / 1e6:.1f} Mbases): fastplong_gpu -w 4 {t2 - t1:.2f} s (device FASTQ parse), "
          f"{t3 - t2:.2f} s (reference reader)")
    assert got_host["out_md5"] == ref["out_md5"] and got_host["json_text_md5"] == ref["json_text_md5"]
    assert got["out_md5"] == ref["out_md5"]
    assert got["failed_md5"] == ref["failed_md5"]
    assert got["json_text_md5"] == ref["json_text_md5"]


def _mutate_fastq(src, dst, kind):
    """Inputs the reference accepts but the device parser does not (FastqReader::getLine / read, src/fastqreader.cpp:219-347)."""
    data = open(src, "rb").read()
    if kind == "crlf":
        data = data.replace(b"\n", b"\r\n")
    elif kind == "blank_line_mid":                     # beyond the pre-scanned head, far from the tail: found mid-run -> restart
        at = data.index(b"\n@read", len(data) // 2) + 1
        data = data[:at] + b"\n" + data[at:]
    elif kind == "cr_mid":
        at = data.index(b"\n+\n", len(data) // 2)
        data = data[:at] + b"\r" + data[at:]
    elif kind == "blank_line_eof":
        data = data + b"\n"
    elif kind == "truncated_last_record":
        data = data[:data.rindex(b"\n+\n") + 3]         # the last record loses its quality line
    elif kind == "stray_line_between_records":
        at = data.index(b"\n@read", len(data) // 2) + 1
        data = data[:at] + b"this line is skipped by the reference\n" + data[at:]
    open(dst, "wb").write(data)


@needs_bin
@pytest.mark.parametrize("kind", ["crlf", "blank_line_mid", "cr_mid", "blank_line_eof", "truncated_last_record",
                                  "stray_line_between_records"])
def test_gpu_binary_non_strict_fastq_like_reference(kind, tmp_path):
    """Drop-in robustness: whatever the reference's reader makes of a non-strict FASTQ, the GPU binary makes the same of
    it (routed to the reference reader up front, or the raw-text run abandoned and restarted) — never a late abort with
    partial outputs."""
    opt = cases.OPTION_SETS["cut_polyx_cplx"]
    batch = synth.ont_like(900, 4000, 77, p_chimera=0.03)
    plain, fq = str(tmp_path / "plain.fq"), str(tmp_path / "in.fq")
    synth.to_fastq(batch, plain)
    _mutate_fastq(plain, fq, kind)
    ref = reference_run(f"non_strict/{kind}", opt, fq, str(tmp_path), 3)
    got = run(GPU_BIN, opt, fq, str(tmp_path), "gpu", 3)
    assert got["out_md5"] == ref["out_md5"]
    assert got["failed_md5"] == ref["failed_md5"]
    assert got["json_text_md5"] == ref["json_text_md5"]


@needs_bin
@pytest.mark.parametrize("emit", ["host", "device"])
@pytest.mark.parametrize("chunk_kb,threads", [(256, 4), (64, 7), (1, 2)])
def test_gpu_binary_many_small_chunks(chunk_kb, threads, emit, tmp_path):
    """The chunk plumbing of the raw-text path (reader -> T workers -> writer's round-robin walk, back-pressure keyed on
    chunk order) with hundreds of chunks: FPL_CHUNK_KB cuts the text into small pieces; 1 KB is smaller than most records,
    so the reader has to keep reading until a record boundary shows up."""
    opt = cases.OPTION_SETS["cut_polyx_cplx"]
    batch = synth.ont_like(2500 if chunk_kb > 1 else 300, 4000, 5 + chunk_kb, p_chimera=0.05, p_polya=0.03, q_mean=17.0)
    fq = str(tmp_path / "in.fq")
    synth.to_fastq(batch, fq)
    env = {"FPL_CHUNK_KB": str(chunk_kb), "FPL_WRITER_BACKLOG": "1"}
    if emit == "device":
        env["FPL_DEVICE_EMIT"] = "1"
    ref = reference_run(f"chunks/{chunk_kb}kb/w{threads}", opt, fq, str(tmp_path), threads)
    got = run(GPU_BIN, opt, fq, str(tmp_path), "gpu", threads, env=env)
    assert got["out_md5"] == ref["out_md5"]
    assert got["failed_md5"] == ref["failed_md5"]
    assert got["json_text_md5"] == ref["json_text_md5"]


@needs_bin
def test_gpu_binary_file_size_is_a_multiple_of_the_chunk(tmp_path):
    """The last fread returns 0 bytes: the final chunk is whatever was left over (possibly nothing)."""
    opt = cases.OPTION_SETS["default_se"]
    batch = synth.ont_like(400, 3000, 12, q_mean=17.0)
    fq = str(tmp_path / "in.fq")
    synth.to_fastq(batch, fq)
    size = os.path.getsize(fq)
    unit = 64 << 10
    pad = (-(size + 27)) % unit          # a last record "@p" + pad x's with 10 bases is pad + 27 bytes long
    with open(fq, "ab") as f:
        f.write(b"@p" + b"x" * pad + b"\nACGTACGTAC\n+\nIIIIIIIIII\n")
    assert os.path.getsize(fq) % unit == 0
    ref = reference_run("chunk_multiple", opt, fq, str(tmp_path), 3)
    got = run(GPU_BIN, opt, fq, str(tmp_path), "gpu", 3, env={"FPL_CHUNK_KB": "64"})
    assert got["out_md5"] == ref["out_md5"]
    assert got["failed_md5"] == ref["failed_md5"]
    assert got["json_text_md5"] == ref["json_text_md5"]


@needs_bin
@pytest.mark.parametrize("emit", ["host", "device"])
def test_gpu_binary_plus_lines_kept_verbatim(emit, tmp_path):
    """The third line of a record may repeat the name ('+name ...'): Read::appendToString writes it back as it was
    (src/read.cpp:119-143), for passing reads, both halves of a split read and --failed_out alike."""
    opt = cases.OPTION_SETS["cut_polyx_cplx"]
    batch = synth.ont_like(600, 3000, 88, p_chimera=0.2, p_polya=0.05, q_mean=16.5)   # ~150 split reads, ~30 failed
    fq = str(tmp_path / "in.fq")
    with open(fq, "wb") as f:
        for i in range(batch.n_reads):
            s, q = batch.read(i)
            name = b"@read%d len=%d" % (i, len(s))
            plus = b"+" if i % 3 == 0 else (b"+" + name[1:] if i % 3 == 1 else b"+ free text %d" % i)
            f.write(name + b"\n" + s + b"\n" + plus + b"\n" + q + b"\n")
    ref = reference_run("plus_lines", opt, fq, str(tmp_path), 3)
    got = run(GPU_BIN, opt, fq, str(tmp_path), "gpu", 3, env={"FPL_DEVICE_EMIT": "1"} if emit == "device" else None)
    assert got["out_md5"] == ref["out_md5"]
    assert got["failed_md5"] == ref["failed_md5"]
    assert got["json_text_md5"] == ref["json_text_md5"]
