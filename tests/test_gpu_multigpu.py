"""Multi-GPU parity on hardware: ONE batch sharded by bases over 2 GPUs (torchrun, one process per GPU), processed
through the C ABI, merged with fpl_allreduce_stats (NCCL on the library's stream), records gathered — compared with a
single pass of the oracle.  Needs two GPUs (run with `gpurun --gpus 2`); skipped on a one-GPU box."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.gpu
@pytest.mark.parametrize("optset", ["cut_polyx_cplx", "default_se"])
def test_two_gpu_shard_merge_gather(optset):
    if _n_gpus() < 2:
        pytest.skip("needs 2 GPUs")
    port = 29600 + os.getpid() % 300
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "mgpu_worker.py"), optset]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-3000:]
    assert "MGPU_OK world=2" in p.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("name,threads,env", [("cut_polyx_cplx", 4, None), ("mask_and_break", 3, {"FPL_DEVICE_EMIT": "1"}),
                                              ("default_se", 5, {"FPL_HOST_PARSE": "1"})])
def test_drop_in_binary_workers_over_two_gpus(name, threads, env, tmp_path):
    """build/fastplong_gpu spreads its worker contexts over the visible devices (worker t -> device t mod 2) and the
    reference's own Stats::merge adds them on the host: outputs and JSON must equal the reference binary's (stored)."""
    if _n_gpus() < 2:
        pytest.skip("needs 2 GPUs")
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    import cases
    import test_gpu_binary as tb
    from fastplong_b200 import synth
    if not os.path.exists(tb.GPU_BIN):
        pytest.skip("build/fastplong_gpu not built")
    opt = cases.OPTION_SETS.get(name) or cases.MASK_BREAK_SETS[name]
    batch = synth.ont_like(3000, 5000, 77, p_chimera=0.03, p_polya=0.03, q_mean=17.0)    # several chunks per worker
    fq = str(tmp_path / "in.fq")
    synth.to_fastq(batch, fq)
    ref = tb.reference_run(f"two_gpus/{name}/w{threads}", opt, fq, str(tmp_path), threads)
    got = tb.run(tb.GPU_BIN, opt, fq, str(tmp_path), "gpu", threads, env=dict(env or {}, FPL_TIMING="1"))
    assert got["out_md5"] == ref["out_md5"]
    assert got["failed_md5"] == ref["failed_md5"]
    assert got["json_text_md5"] == ref["json_text_md5"]
