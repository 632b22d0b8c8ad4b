"""Gzip output on the device (fpl_gzip_host, fpl_emit_fastq_gzip_host, FPL_DEVICE_GZIP=1 in the drop-in CLI).  Python's
zlib / gzip is the independent decoder: it checks every member's CRC-32 and ISIZE and raises on any error.  Only the
decompressed content is pinned, never the compressed bytes of another encoder."""
import ctypes as C
import gzip
import hashlib
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

import cases
from fastplong_b200 import abi, synth
from test_gpu_binary import GPU_BIN, _mutate_fastq, json_text_md5, needs_bin
from test_gpu_emit import fastq_of

pytestmark = pytest.mark.gpu

SEG = abi.GZIP_SEGMENT
EMULATE = os.environ.get("FPL_EMULATE", "") not in ("", "0")


def engine(opt=None):
    from fastplong_b200 import Options
    from fastplong_b200.binding import Engine
    return Engine(opt or Options())


def members(data):
    """The decompressed members of a multi-member gzip stream, in order."""
    out = []
    while data:
        d = zlib.decompressobj(31)
        out.append(d.decompress(data) + d.flush())
        assert d.eof, "truncated gzip member"
        data = d.unused_data
    return out


def short_name_fastq():
    b = synth.ont_like(3000, 4000, 7)
    return b"".join(b"@read%d len=%d\n%s\n+\n%s\n" % (i, len(b.read(i)[0]), *b.read(i)) for i in range(b.n_reads))


def ont_header_fastq():
    """The same reads behind realistic ONT header lines (UUID, runid=, start_time= ...), from a seeded generator."""
    b = synth.ont_like(3000, 4000, 7)
    rng = np.random.default_rng(3)
    parts = []
    for i in range(b.n_reads):
        u = rng.integers(0, 256, 16, dtype=np.uint8).tobytes().hex()
        name = (b"@%s-%s-%s-%s-%s runid=8f3e2b7c9d4a1e6f0b5c2d8e7a9f1c3b4d6e8a0b read=%d ch=%d "
                b"start_time=2024-03-%02dT%02d:%02d:%02dZ flow_cell_id=PAK12345 protocol_group_id=run1 sample_id=sample1 "
                b"barcode=barcode%02d" % (u[:8].encode(), u[8:12].encode(), u[12:16].encode(), u[16:20].encode(),
                                          u[20:].encode(), i, rng.integers(1, 513), rng.integers(1, 28), rng.integers(0, 24),
                                          rng.integers(0, 60), rng.integers(0, 60), rng.integers(1, 25)))
        parts.append(name + b"\n%s\n+\n%s\n" % b.read(i))
    return b"".join(parts)


def inputs():
    rng = np.random.default_rng(11)
    mib = 1 << 20
    yield "empty", b""
    yield "one_byte", b"x"
    for n in (SEG - 1, SEG, SEG + 1):
        yield f"text_{n}", bytes(rng.integers(32, 127, n, dtype=np.uint8))
    yield "random", rng.integers(0, 256, mib, dtype=np.uint8).tobytes()
    yield "all_A", b"A" * mib
    for period in (1, 2, 3, 7, 31, 64, 255, 258, 259, 300):
        unit = rng.integers(0, 256, period, dtype=np.uint8).tobytes()
        yield f"period_{period}", (unit * (mib // period + 1))[:mib]
    yield "every_byte", bytes(range(256)) * (mib // 256)
    yield "fastq_short_names", short_name_fastq()[:mib]
    yield "fastq_ont_headers", ont_header_fastq()[:mib]


INPUTS = dict(inputs())


@pytest.fixture(scope="module")
def eng():
    return engine()


@pytest.mark.parametrize("name", sorted(INPUTS))
def test_round_trip_and_bound(eng, name):
    x = INPUTS[name]
    out = eng.gzip([x])
    assert len(out) == 1
    z = out[0]
    if not x:
        assert z == b""
        return
    assert gzip.decompress(z) == x
    ms = members(z)
    assert len(ms) == -(-len(x) // SEG)
    assert ms == [x[i:i + SEG] for i in range(0, len(x), SEG)]
    assert z[:10] == bytes([0x1f, 0x8b, 8, 0, 0, 0, 0, 0, 0, 0xff])
    assert len(z) <= abi.gzip_bound(len(x), 1)


def test_random_input_grows_by_the_stored_overhead_only(eng):
    x = INPUTS["random"]
    z = eng.gzip([x])[0]
    segs = -(-len(x) // SEG)
    assert len(z) <= len(x) + segs * (10 + 8 + 2 * 5)


def test_many_pieces_with_empty_ones(eng):
    rng = np.random.default_rng(5)
    sizes = [0, 1, 0, SEG, 3 * SEG + 17, 0, 1000, SEG - 1, 0]
    pieces = [rng.integers(60, 80, n, dtype=np.uint8).tobytes() for n in sizes]
    out = eng.gzip(pieces)
    assert len(out) == len(pieces)
    for p, z in zip(pieces, out):
        if not p:
            assert z == b""
        else:
            assert gzip.decompress(z) == p
            assert len(members(z)) == -(-len(p) // SEG)
    assert eng.gzip([]) == []
    assert sum(map(len, out)) <= abi.gzip_bound(sum(sizes), len(sizes))


def test_too_small_output_buffer_fails(eng):
    from fastplong_b200.binding import FplError
    x = np.frombuffer(b"ACGT" * 1000, dtype=np.uint8)
    sizes = np.array([x.size], dtype=np.int64)
    cap = abi.gzip_bound(x.size, 1) - 1
    out = np.zeros(cap, dtype=np.uint8)
    osz = np.zeros(1, dtype=np.int64)
    rc = eng.lib.fpl_gzip_host(eng.h, x.ctypes.data, sizes.ctypes.data, 1, out.ctypes.data, cap, osz.ctypes.data)
    assert rc < 0
    with pytest.raises(FplError):
        eng._check(rc)


@pytest.mark.parametrize("corpus", ["short_names", "ont_headers"])
def test_ratio_against_zlib_level_4(eng, corpus):
    x = short_name_fastq() if corpus == "short_names" else ont_header_fastq()
    z = eng.gzip([x])[0]
    assert gzip.decompress(z) == x
    ratio = len(z) / len(zlib.compress(x, 4))
    print(f"\n{corpus}: {len(x)} bytes -> {len(z)} bytes, {ratio:.4f} x zlib level 4")
    assert ratio <= 1.08


def _digest(eng):
    h = hashlib.sha256()
    for name in sorted(INPUTS):
        if len(INPUTS[name]) <= 2 * SEG or name.startswith(("fastq", "period_3", "all_A")):
            for z in eng.gzip([INPUTS[name], INPUTS[name][:1000]]):
                h.update(z)
    return h.hexdigest()


def test_deterministic(eng):
    d = _digest(eng)
    assert _digest(eng) == d
    assert _digest(engine()) == d
    if EMULATE:
        # the emulated run with the threads of every block scheduled in a random order gives the same bytes
        code = ("import sys; sys.path[:0] = %r; import conftest, simt_emu; from fastplong_b200 import binding; "
                "binding.LIB_PATH = simt_emu.build_library(); import test_gpu_gzip as t; print(t._digest(t.engine()))"
                % [os.path.dirname(os.path.dirname(os.path.abspath(__file__))), os.path.dirname(os.path.abspath(__file__))])
        for seed in (1, 2):
            r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=1200,
                               env=dict(os.environ, EMU_SCHED=f"random:{seed}"))
            assert r.returncode == 0, r.stderr[-2000:]
            assert r.stdout.split()[-1] == d


EMIT_CASES = [("default_se", lambda: cases.ont_batch(91, n=400, mean=2500, p_chimera=0.2)),
              ("cut_polyx_cplx", lambda: cases.ont_batch(92, n=300, mean=1500, p_chimera=0.1)),
              ("trims_limits", lambda: cases.adversarial_batch(3))]
EMIT_CASES += [(name, lambda: cases.blocky_quality_batch(77)) for name in sorted(cases.MASK_BREAK_SETS)]


@pytest.mark.parametrize("name,make", EMIT_CASES, ids=[c[0] for c in EMIT_CASES])
@pytest.mark.parametrize("want_failed", [True, False])
def test_emit_gzip_matches_emit(name, make, want_failed):
    opt = cases.OPTION_SETS.get(name) or cases.MASK_BREAK_SETS[name]
    text, _, _ = fastq_of(make())
    g = engine(opt)
    assert g.process_fastq(text) is not None
    zo, zf = g.emit_fastq_gzip(want_failed)
    out, failed = g.emit_fastq(want_failed)
    assert (gzip.decompress(zo) if zo else b"") == out
    assert (gzip.decompress(zf) if zf else b"") == failed
    assert g.emit_fastq_gzip(want_failed) == (zo, zf)             # the compressed text stays built
    assert len(zo) <= abi.gzip_bound(len(out), 1) and len(zf) <= abi.gzip_bound(len(failed), 1)


def test_emit_gzip_too_small_buffer_copies_nothing():
    opt = cases.OPTION_SETS["cut_polyx_cplx"]
    text, _, _ = fastq_of(cases.ont_batch(93, n=200, mean=2000, p_chimera=0.1))
    g = engine(opt)
    g.process_fastq(text)
    n_out, n_failed = C.c_int64(), C.c_int64()
    rc = g.lib.fpl_emit_fastq_gzip_host(g.h, 1, None, 0, C.byref(n_out), None, 0, C.byref(n_failed))
    assert rc == 1 and n_out.value > 0
    out = np.full(n_out.value - 1, 0xAB, dtype=np.uint8)
    failed = np.full(max(n_failed.value, 1), 0xAB, dtype=np.uint8)
    rc = g.lib.fpl_emit_fastq_gzip_host(g.h, 1, out.ctypes.data, out.size, C.byref(n_out), failed.ctypes.data, failed.size,
                                        C.byref(n_failed))
    assert rc == 1
    assert (out == 0xAB).all() and (failed == 0xAB).all()
    zo, zf = g.emit_fastq_gzip(True)
    assert (gzip.decompress(zo), gzip.decompress(zf)) == g.emit_fastq(True)


# ---- the drop-in CLI: FPL_DEVICE_GZIP=1 ----
def run_cli(opt, fq, outdir, tag, threads, env=None, gz=True, extra=()):
    sfx = ".fq.gz" if gz else ".fq"
    out, failed, js, html = (os.path.join(outdir, f"{tag}.{n}") for n in ("o" + sfx, "f" + sfx, "json", "html"))
    cmd = [GPU_BIN, "-i", fq, "-o", out, "--failed_out", failed, "-j", js, "-h", html, "-w", str(threads)]
    cmd += opt.cli_flags() + list(extra)
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ, **(env or {})))
    assert r.returncode == 0, r.stderr[-2000:]
    text = {k: open(p, "rb").read() for k, p in (("out", out), ("failed", failed))}
    if gz:
        text = {k: gzip.decompress(v) if v else b"" for k, v in text.items()}
    return {"out_md5": hashlib.md5(text["out"]).hexdigest(), "failed_md5": hashlib.md5(text["failed"]).hexdigest(),
            "json_text_md5": json_text_md5(js), "out_path": out}


CLI_MODES = {"raw_text": {}, "raw_text+emit": {"FPL_DEVICE_EMIT": "1"}, "chunk64": {"FPL_CHUNK_KB": "64"},
             "gz_input": {}, "non_strict": {}}


@needs_bin
@pytest.mark.parametrize("threads", [1, 3])
@pytest.mark.parametrize("mode", sorted(CLI_MODES))
def test_cli_device_gzip_matches_plain_output(mode, threads, tmp_path):
    opt = cases.OPTION_SETS["cut_polyx_cplx"]
    batch = synth.ont_like(900, 4000, 61 + threads, p_chimera=0.05, p_polya=0.03, q_mean=17.0)
    fq = str(tmp_path / "in.fq")
    synth.to_fastq(batch, fq)
    if mode == "gz_input":                               # the reference reader (reader path)
        data = open(fq, "rb").read()
        fq = str(tmp_path / "in.fq.gz")
        with gzip.open(fq, "wb", compresslevel=1) as f:
            f.write(data)
    elif mode == "non_strict":                           # raw-text run abandoned mid-file and restarted
        src, fq = fq, str(tmp_path / "mut.fq")
        _mutate_fastq(src, fq, "blank_line_mid")
    env = CLI_MODES[mode]
    plain = run_cli(opt, fq, str(tmp_path), "plain", threads, env=env, gz=False)
    dev = run_cli(opt, fq, str(tmp_path), "dev", threads, env=dict(env, FPL_DEVICE_GZIP="1"))
    host = run_cli(opt, fq, str(tmp_path), "host", threads, env=env)        # the writer's own compression, untouched
    for got in (dev, host):
        assert got["out_md5"] == plain["out_md5"]
        assert got["failed_md5"] == plain["failed_md5"]
        assert got["json_text_md5"] == plain["json_text_md5"]
    if mode == "raw_text" and threads == 3:
        # the device-written .gz, read back as input, gives the report the plain file gives
        again_gz = run_cli(cases.OPTION_SETS["default_se"], dev["out_path"], str(tmp_path), "again_gz", 2, gz=False)
        again = run_cli(cases.OPTION_SETS["default_se"], plain["out_path"], str(tmp_path), "again", 2, gz=False)
        assert again_gz["out_md5"] == again["out_md5"]
        assert again_gz["json_text_md5"] == again["json_text_md5"]
