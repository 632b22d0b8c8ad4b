"""Measures gzip output on the device against the host path it replaces, and writes one JSON file.

  python tools/bench_gzip.py --out profiles/gzip_bench.json [--gb 1] [--cli-gb 4] [--repeats 3] [--workdir /tmp]

Records, with the GPU's name and power limit (read-only nvidia-smi query) and the host CPU model taken in the same run:
  * k_gzip_deflate + k_gzip_compact device time per GB of input (fpl_last_kernel_times), on --gb GB of ONT-like FASTQ
    (a 64 MiB seeded corpus repeated: segments are compressed independently, so the repetition does not help the encoder);
  * fpl_gzip_host end to end (host -> device copy, kernels, device -> host copy) in GB/s;
  * Python zlib at level 4 on one thread over 64 MiB of the same text, in MB/s, and both compressed sizes;
  * build/fastplong_gpu --out x.fq.gz wall time with and without FPL_DEVICE_GZIP=1, on a --cli-gb GB plain FASTQ and on a
    gzipped copy of it, alternating the two settings --repeats times; outputs go to --workdir (local disk).
"""
import argparse
import gzip
import json
import os
import platform
import shutil
import subprocess
import sys
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def cpu_model():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return platform.processor() or "unknown"


def corpus(n_bytes, seed=7):
    """ONT-like FASTQ (synth.ont_like, names `@read<i> len=<L>`), at least n_bytes long."""
    from fastplong_b200 import synth
    b = synth.ont_like(max(1, n_bytes // 8000 + 1), 4000, seed)
    text = b"".join(b"@read%d len=%d\n%s\n+\n%s\n" % (i, len(b.read(i)[0]), *b.read(i)) for i in range(b.n_reads))
    return text


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--gb", type=float, default=1.0)
    ap.add_argument("--cli-gb", type=float, default=4.0)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--workdir", default="/tmp")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_gzip: no CUDA device (this measurement has no CPU fallback)")
    from fastplong_b200 import Options
    from fastplong_b200.binding import Engine
    res = {"gpu": gpu_info(), "cpu": cpu_model(), "host_threads": os.cpu_count()}

    base = corpus(64 << 20)[:64 << 20]
    reps = max(1, int(a.gb * (1 << 30)) // len(base))
    text = base * reps
    res["device_input_bytes"] = len(text)
    g = Engine(Options())
    g.gzip([base[:4 << 20]])                                 # warm-up: module load, buffer growth
    g.gzip([text])
    g.set_timing(True)
    t0 = time.perf_counter()
    z = g.gzip([text])[0]
    wall = time.perf_counter() - t0
    kt = g.kernel_times()
    dev_ms = sum(kt[k][0] for k in ("k_gzip_deflate", "k_gzip_compact"))
    gb = len(text) / 1e9
    res["kernel_ms"] = {k: kt[k][0] for k in ("k_gzip_deflate", "k_gzip_compact")}
    res["kernel_ms_per_gb"] = dev_ms / gb
    res["kernel_gb_per_s"] = gb / (dev_ms / 1e3)
    res["fpl_gzip_host_s"] = wall
    res["fpl_gzip_host_gb_per_s"] = gb / wall
    res["device_compressed_bytes"] = len(z)
    assert zlib.decompressobj(31).decompress(z[:1 << 20])        # a decodable start; the test suite checks every byte

    t0 = time.perf_counter()
    z4 = zlib.compress(base, 4)
    res["zlib4_mb_per_s_one_thread"] = len(base) / 1e6 / (time.perf_counter() - t0)
    res["zlib4_ratio_64mib"] = len(base) / len(z4)
    zd = g.gzip([base])[0]
    res["device_ratio_64mib"] = len(base) / len(zd)
    res["device_size_vs_zlib4"] = len(zd) / len(z4)
    g.close()

    binary = os.path.join(ROOT, "build", "fastplong_gpu")
    if a.cli_gb > 0 and os.path.exists(binary):
        wd = os.path.join(a.workdir, "fpl_bench_gzip_%d" % os.getpid())
        os.makedirs(wd, exist_ok=True)
        try:
            fq = os.path.join(wd, "in.fq")
            with open(fq, "wb") as f:
                for _ in range(max(1, int(a.cli_gb * (1 << 30)) // len(base))):
                    f.write(base)
            fqgz = fq + ".gz"
            t0 = time.perf_counter()
            with open(fq, "rb") as src, gzip.open(fqgz, "wb", compresslevel=1) as dst:
                shutil.copyfileobj(src, dst, 16 << 20)
            res["cli_input_bytes"] = os.path.getsize(fq)
            res["cli_gz_input_bytes"] = os.path.getsize(fqgz)
            runs = {}
            for _ in range(a.repeats):
                for inp, name in ((fq, "plain_input"), (fqgz, "gz_input")):
                    for knob in (False, True):
                        out = os.path.join(wd, "x.fq.gz")
                        env = dict(os.environ)
                        env.pop("FPL_DEVICE_GZIP", None)
                        if knob:
                            env["FPL_DEVICE_GZIP"] = "1"
                        cmd = [binary, "-i", inp, "-o", out, "-j", os.path.join(wd, "r.json"), "-h", os.path.join(wd, "r.html"),
                               "-w", "8"]
                        t0 = time.perf_counter()
                        r = subprocess.run(cmd, capture_output=True, text=True, env=env)
                        dt = time.perf_counter() - t0
                        if r.returncode != 0:
                            raise SystemExit(r.stderr[-2000:])
                        key = "%s/%s" % (name, "device_gzip" if knob else "writer_libdeflate")
                        runs.setdefault(key, []).append(dt)
                        runs.setdefault(key + "/out_bytes", []).append(os.path.getsize(out))
                        os.remove(out)
            res["cli_wall_s"] = runs
            res["cli_threads"] = 8
        finally:
            shutil.rmtree(wd, ignore_errors=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    json.dump(res, open(a.out, "w"), indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
