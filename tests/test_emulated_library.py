"""The whole product without a GPU: tests/simt_emu.py builds every .cu of fastplong_b200/csrc (fpl_api.cu's C ABI and host logic
included, fpl_jit.cu compiling its generated source through an NVRTC stand-in) for the host behind the SIMT emulator, and links
host/seprocessor_gpu.cpp with the reference's objects against it.  Here: the emulated library exports the whole C ABI and is
bit-exact against the oracle through binding.Engine (packed batch, FASTQ text in / text out), and the emulated drop-in binary
produces the reference binary's files.  `FPL_EMULATE=1 python -m pytest tests -m gpu` runs the GPU test files on the same build."""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np
import pytest

import cases
import simt_emu
from fastplong_b200 import binding, hostside, synth
from oracle_lib import REF_BIN, OracleEngine, compare_results, compare_stats
from test_abi_exports import header_functions


@pytest.fixture()
def emulated_binding():
    """binding.Engine on the emulated library for the duration of one test"""
    with simt_emu._Bound() as b:
        yield b


def test_emulated_library_exports_the_c_abi():
    lib = C.CDLL(simt_emu.build_library())
    for name in header_functions():
        assert hasattr(lib, name), name


def test_engine_on_the_emulated_library_is_bit_exact(emulated_binding, capfd):
    opt = cases.OPTION_SETS["cut_polyx_cplx"]
    batch = synth.ont_like(80, 2500, 123, p_chimera=0.1, p_polya=0.05)
    g, o = emulated_binding.Engine(opt), OracleEngine(opt)
    res = g.process(batch)
    compare_results(res, o.process(batch), "emulated library")
    cyc = int(batch.lens.max())
    for w in (0, 1):
        compare_stats(g.stats(w, cyc), o.stats(w, cyc), f"emulated library/stats{w}")
    compare_stats(g.counters(), o.counters(), "emulated library/counters")
    assert g.launch_count >= 13
    g.close()
    assert "specialisation unavailable" not in capfd.readouterr().err        # fpl_jit.cu built k_scan_jit through the NVRTC stand-in


def test_fastq_text_through_the_emulated_c_abi(emulated_binding):
    opt = cases.MASK_BREAK_SETS["mask_and_break"]
    batch = cases.blocky_quality_batch(5, n=40)
    names = [b"@read%d len=%d" % (i, int(batch.lens[i])) for i in range(batch.n_reads)]
    text = b"".join(nm + b"\n" + batch.read(i)[0] + b"\n+\n" + batch.read(i)[1] + b"\n" for i, nm in enumerate(names))
    g, o = emulated_binding.Engine(opt), OracleEngine(opt)
    recs, res, used = g.process_fastq(text)
    assert used == len(text) and len(recs) == batch.n_reads
    ores = o.process(batch)
    compare_results(res, ores, "emulated text path")
    out, failed = g.emit_fastq(True)
    exp_out, exp_failed = hostside.emit_fastq_ext(batch, names, ores, o.segments(), o.mask_regions())
    assert out == exp_out and failed == exp_failed
    g.close()


@pytest.mark.skipif(not os.path.exists(REF_BIN) or not os.path.exists(os.path.join(simt_emu.ROOT, "oracle", "_ref", "obj", "main.o"))
                    or not simt_emu.REF_SRC or not os.path.exists(os.path.join(simt_emu.REF_SRC, "main.cpp")),
                    reason="oracle/_ref (the reference's objects and binary) not built, or the reference's headers absent")
@pytest.mark.parametrize("flags,threads", [(["--cut_front", "--cut_tail", "-x", "-y"], 3), (["-N", "-b", "-s", synth.ADAPTER_START], 2)])
def test_emulated_drop_in_binary_writes_the_reference_binary_s_files(flags, threads, tmp_path):
    exe = simt_emu.build_binary()
    fq = str(tmp_path / "in.fq")
    synth.to_fastq(synth.ont_like(400, 2500, 9, p_chimera=0.1, p_polya=0.1, q_mean=16.0), fq)
    md5 = {}
    for name, binary in (("ref", REF_BIN), ("emu", exe)):
        d = str(tmp_path / name)
        os.makedirs(d)
        r = subprocess.run([binary, "-i", fq, "-o", d + "/o.fq", "--failed_out", d + "/f.fq", "-j", d + "/j.json", "-h", d + "/h.html",
                            "-w", str(threads)] + flags, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-1500:]
        js = b"\n".join(ln for ln in open(d + "/j.json", "rb").read().split(b"\n") if b'"command"' not in ln)
        md5[name] = [hashlib.md5(x).hexdigest() for x in (open(d + "/o.fq", "rb").read(), open(d + "/f.fq", "rb").read(), js)]
        assert os.path.getsize(d + "/o.fq") > 50000
    assert md5["emu"] == md5["ref"]


def test_limits_of_the_c_abi_on_the_emulated_library():
    """FPL_MAX_ADAPTERS and FPL_MAX_ADAPTER_LEN: the largest accepted adapter set works (1022 FASTA entries + -s / -e, bit-exact),
    one more entry or one more base is a loud error of fpl_create"""
    from fastplong_b200 import Options
    from test_simt_kernels import check
    rng = np.random.default_rng(1)
    ad = lambda n: "".join("ACGT"[i] for i in rng.integers(0, 4, size=n))
    fa = sorted(ad(int(rng.integers(8, 30))) for _ in range(1022))
    check(Options(start_adapter=synth.ADAPTER_START, end_adapter=synth.ADAPTER_END, adapter_fasta=fa), cases.ont_batch(3, n=6, mean=800), "1022 adapters")
    with pytest.raises(binding.FplError, match="FPL_MAX_ADAPTERS"):
        simt_emu.EmuEngine(Options(adapter_fasta=fa + [ad(10)]))
    with pytest.raises(binding.FplError, match="FPL_MAX_ADAPTER_LEN"):
        simt_emu.EmuEngine(Options(start_adapter=ad(1025)))
