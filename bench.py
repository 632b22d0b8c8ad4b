#!/usr/bin/env python
"""bench.py — Gbases/s of fastplong's per-read hot loop (adapter-trim + Q-filter + stats) on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): 1M DISTINCT ONT-like reads, mean 15 kb (32 GB of payload, generated on the
device), adapters as the reference's evaluator auto-detects them on this generator's reads, --cut_front --cut_tail
-W 10, default Q/length filters, pre+post Stats.  Before anything is timed the first reads of the input go through
the GPU library and the CPU oracle and are compared word by word (`parity_checked`); behind the timed legs the whole
batch is checked once more at full size (`parity_full_scale`: records of read ranges spread over the 32 GB against the
oracle, every word of both Stats blocks against an independent torch restatement — full_scale_check below).
One step = one pass of processSingleEnd over the whole per-GPU batch (+ the Stats/FilterResult all-reduce when N>1).
`value` = device-resident throughput; `e2e` = the same metric through fpl_process_host with pinned HOST buffers
(H2D of every byte + D2H of the per-read records inside the timed region).
--dump-outputs DIR writes what the last timed step computed as DIR/<name>.npy (float64, exact): both Stats blocks, the
FilterResult counters and the per-read records of a fixed, seeded sample of the reads.  The inputs depend on the arguments
only, so two builds can be compared file by file.

--impl reference times the reference's own CPU implementation (oracle/_ref/fastplong_ref, built from the
unmodified sources) on a bounded sample of the same workload with all host threads it can use.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

MEAN_LEN = 15000
SEED = 20260924
ALG_BYTES_PER_BASE = 2      # 1 sequence byte + 1 quality byte, each read once (SURVEY §8d)
ALG_BYTES_PER_READ = 64     # offset, length, result record
HBM_FALLBACK_GBS = 6650.0   # /opt/skills/guides/B200_PROFILING.md fallback
# CPU arm: a sample large enough that the binary's fixed costs (start-up, adapter detection pre-pass, report writing)
# do not dominate: 40k reads x 15 kb = 0.6 Gbases, a few seconds of reference CPU time per run with 16 workers
REF_SAMPLE_READS = int(os.environ.get("FPL_BENCH_REF_READS", "40000"))   # the override exists for the CPU test of this arm
PARITY_BASES = int(os.environ.get("FPL_BENCH_PARITY_BASES", "60000000"))   # the slice compared with the oracle outside the timed region (a few seconds of CPU)
FULL_CHECK_RANGES = 8       # read ranges spread over the whole batch whose records are compared with the oracle ...
FULL_CHECK_BASES = 24_000_000   # ... this many bases in total
FULL_CHECK_BUDGET_S = 150   # the torch restatement of the Stats blocks gives up beyond this (reported, not fatal)
E2E_SUBMISSIONS = 64        # host submissions per step of the end-to-end leg
E2E_HOST_CHUNKS = 4         # distinct pinned host chunks cycled through them
DUMP_BYTES = 64 << 20       # --dump-outputs: at most this much in all
DUMP_MAX_READS = 1 << 17    # ... and the records of at most this many reads


# name: (reads per GPU, replicas, mean length, generator keywords, description)
WORKLOADS = {
    "c2": (1 << 20, 1, MEAN_LEN, {},
           "configs[1]: 1M ONT reads mean 15 kb, auto-detected adapters + --cut_front --cut_tail -W 10, default filters, "
           "pre+post stats"),
    "c3": (625_000, 1, 20000, dict(q_mean=33.0, q_sd=6.0, q_clip=60, p_polya=0.05, p_planted=0.2),
           "configs[2], one GPU's share of an 8-GPU run (5M / 8 = 625k PacBio-HiFi-like reads mean 20 kb; the whole set "
           "is 200 GB and does not fit one GPU): --adapter_fasta 64-entry set + polyX trim"),
    "c4": (2_500_000, 1, 10000, {},
           "configs[3], one GPU's share (20M / 8 = 2.5M ONT reads mean 10 kb): full pipeline — adapters + Q filter + "
           "length filter (--length_required 1000 --length_limit 60000) + low-complexity filter (-y) + pre/post stats"),
    "c5-1k": (100_000, 1, 1000, dict(min_len=100), "configs[4]: 100k reads mean 1 kb, adapter trim only (-Q -L)"),
    "c5-50k": (100_000, 1, 50000, {}, "configs[4]: 100k reads mean 50 kb, adapter trim only (-Q -L)"),
    "c5-500k": (20_000, 1, 500000, {}, "configs[4] at 1/5 of the read count (20k reads mean 500 kb = 10 Gbases; 100k would be "
                                       "100 GB of payload): adapter trim only (-Q -L)"),
}


def c3_fasta():
    rng = np.random.default_rng(64)
    return sorted("".join("ACGT"[i] for i in rng.integers(0, 4, size=int(rng.integers(20, 45)))) for _ in range(64))


def workload_options(name="c2"):
    from fastplong_b200 import Options, synth
    if name == "c3":
        return Options(start_adapter=synth.ADAPTER_START, end_adapter=synth.ADAPTER_END, adapter_fasta=c3_fasta(),
                       trim_poly_x=True)
    if name == "c4":
        return Options(start_adapter=synth.ADAPTER_START, end_adapter=synth.ADAPTER_END, low_complexity_filter=True,
                       length_required=1000, length_limit=60000)
    if name.startswith("c5"):
        return Options(start_adapter=synth.ADAPTER_START, end_adapter=synth.ADAPTER_END, disable_quality_filtering=True,
                       disable_length_filtering=True)
    # -s/-e left at "auto" on the CLI; the strings below are what Evaluator::evalAdapterAndReadNum detects on this
    # generator's reads (verified with oracle/_ref/fastplong_ref, DESIGN.md §Measurement) — the pre-pass itself is
    # outside the hot path (SURVEY §8d).
    return Options(start_adapter=synth.ADAPTER_START, end_adapter=synth.ADAPTER_END, cut_front=True, cut_tail=True,
                   cut_window_size=10)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons during the timed region (pynvml)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._halt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if not self.nv:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._halt.wait(0.05)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


def physical_device_index(local):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local])
        except Exception:
            return local
    return local


def parity_check(opt, host_slice):
    """One slice of the bench input through the GPU library and through the CPU oracle (the checker, outside every timed
    region): per-read records, both Stats blocks and the counters, word by word.  Raises on the first difference."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from fastplong_b200.binding import Engine
    from oracle_lib import OracleEngine, compare_results, compare_stats
    gpu = Engine(opt)
    res = gpu.process(host_slice)
    orc = OracleEngine(opt)
    ref = orc.process(host_slice)
    compare_results(res, ref, "bench parity slice")
    cyc = int(host_slice.lens.max())
    for w in (0, 1):
        compare_stats(gpu.stats(w, cyc), orc.stats(w, cyc), f"bench parity slice/stats{w}")
    compare_stats(gpu.counters(), orc.counters(), "bench parity slice/counters")
    gpu.close()
    orc.close()
    return {"reads": host_slice.n_reads, "bases": host_slice.n_bases,
            "compared": "records field by field, pre and post Stats blocks and FilterResult counters word by word, GPU library vs "
                        "the C oracle (oracle/fpl_oracle.c) on the first reads of this run's input, outside the timed region"}


def full_scale_check(torch, eng, opt, tile, d_seq, d_qual, offsets, lens, tile_reads, mean_len, budget_s=FULL_CHECK_BUDGET_S):
    """Parity at the size the number is quoted on, outside every timed region, on what the LAST device-resident pass over
    the whole batch left in the context (the caller has just run one):
    (1) the records of FULL_CHECK_RANGES read ranges spread over the batch — the last one ends with the last read, tens
        of GB into the buffers — against the C oracle run on exactly those reads;
    (2) every word of the pre- and post-filter Stats blocks, and every read's / passing segment's median quality, against
        tests/stats_tables.py: an independent restatement of Stats::statRead as torch.bincount passes over the same
        device buffers (pinned to the oracle on the CPU by tests/test_stats_tables.py);
    (3) the FilterResult counters against the records (one filter result per segment, passing segments = post reads).
    Raises AssertionError on the first difference; returns what was compared."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from fastplong_b200 import abi
    from oracle_lib import OracleEngine, compare_results
    from stats_tables import passing_segments, stats_block
    t0 = time.time()
    offsets = np.asarray(offsets, dtype=np.int64)
    lens = np.asarray(lens)
    n_reads = len(lens)
    res = eng.fetch_results(n_reads)
    out = {"reads": n_reads, "bases": int(lens.sum(dtype=np.int64))}
    # (1) sampled records
    m = int(min(tile_reads, max(4, FULL_CHECK_BASES // FULL_CHECK_RANGES // max(1, mean_len))))
    n_cmp = b_cmp = 0
    spans = []
    for j in range(1, FULL_CHECK_RANGES + 1):
        g1 = max(1, n_reads * j // FULL_CHECK_RANGES)
        rep = (g1 - 1) // tile_reads                       # keep a range inside one replica of the tile
        hi_t = g1 - rep * tile_reads
        lo_t = max(0, hi_t - m)
        g0 = rep * tile_reads + lo_t
        hb = tile.to_host(lo_t, hi_t)
        orc = OracleEngine(opt)
        ref = orc.process(hb)
        orc.close()
        compare_results(res[g0:g1], ref, f"full-scale records, reads [{g0}, {g1}) at byte {int(offsets[g0])}")
        n_cmp += g1 - g0
        b_cmp += hb.n_bases
        spans.append([int(g0), int(g1)])
    out["records_vs_oracle"] = {"reads": n_cmp, "bases": b_cmp, "read_ranges": spans,
                                "highest_byte_offset": int(offsets[n_reads - 1])}
    # (3) counters against the records
    cnt = eng.counters()
    rd, k, starts, seg_lens = passing_segments(res, offsets)
    assert int(cnt[abi.CNT_FILTER:abi.CNT_FILTER + 32].sum()) == int(res["n_segments"].sum()), "filter results != segments"
    assert int(cnt[abi.CNT_FILTER + abi.PASS_FILTER]) == len(rd), "passed counter != passing segments"
    # (2) Stats blocks
    cap = eng.cycles
    deadline = t0 + budget_s
    for which, (st, ln, medians, nz) in enumerate(((offsets, lens.astype(np.int64), res["pre_median_qual"], lens > 0),
                                                   (starts, seg_lens, res["seg_median_qual"][rd, k], seg_lens > 0))):
        blk, med = stats_block(torch, d_seq, d_qual, st, ln, cap, deadline=deadline)
        got = eng.stats(which)
        if not np.array_equal(blk, got):
            bad = np.nonzero(blk != got)[0]
            raise AssertionError(f"full-scale Stats block {which}: {len(bad)} words differ, first at {int(bad[0])}: "
                                 f"{int(got[bad[0]])} (library) vs {int(blk[bad[0]])} (torch restatement)")
        if not np.array_equal(med[nz], medians[nz]):
            raise AssertionError(f"full-scale medians of Stats block {which} differ on {int((med[nz] != medians[nz]).sum())} segments")
    out["stats_vs_torch"] = {"blocks": ["pre", "post"], "words_each": int(abi.stats_words(cap)), "passing_segments": int(len(rd)),
                             "medians": "every read (pre) and every passing segment (post)"}
    out["ok"] = True
    out["seconds"] = round(time.time() - t0, 1)
    out["compared"] = ("after one more untimed device-resident pass over the whole batch: records of %d read ranges spread over the "
                       "buffers vs the C oracle; every word of both Stats blocks and every median vs an independent torch.bincount "
                       "restatement of Stats::statRead over the same device buffers (tests/stats_tables.py); FilterResult counters "
                       "vs the records" % FULL_CHECK_RANGES)
    return out


def dump_outputs(eng, n_reads, cycles, out_dir):
    """What the caller of the timed path receives after a step: both Stats blocks (laid out over the longest read's
    cycles), the counters and the per-read records, one .npy per field.  The records are those of a fixed, seeded sample
    of the reads (sorted read indices in records_read_index.npy) sized so that everything stays within DUMP_BYTES; a Stats
    block above 3/8 of DUMP_BYTES (reads of hundreds of kb) is cut to a fixed, seeded sample of its words the same way."""
    from fastplong_b200.abi import RESULT_DTYPE
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"counters": eng.counters()}
    for which, name in ((0, "stats_pre"), (1, "stats_post")):
        block = eng.stats(which, cycles)
        if block.size * 8 > DUMP_BYTES * 3 // 8:
            arrays[name + "_index"] = np.sort(np.random.default_rng(SEED + which).choice(block.size, DUMP_BYTES // 64,
                                                                                          replace=False))
            block = block[arrays[name + "_index"]]
        arrays[name] = block
    fixed = sum(a.size for a in arrays.values()) * 8
    per_read = 8 * (1 + sum(int(np.prod(RESULT_DTYPE[f].shape or (1,))) for f in RESULT_DTYPE.names))
    k = int(min(n_reads, DUMP_MAX_READS, max(0, DUMP_BYTES - fixed) // per_read))
    idx = np.sort(np.random.default_rng(SEED).choice(n_reads, size=k, replace=False)) if k < n_reads else np.arange(n_reads)
    res = eng.fetch_results(n_reads)[idx]
    arrays["records_read_index"] = idx
    for f in RESULT_DTYPE.names:
        arrays["records_" + f] = res[f]
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))
    return {"dir": out_dir, "files": len(arrays), "sampled_reads": k,
            "bytes": int(sum(np.asarray(a).size for a in arrays.values()) * 8)}


def h2d_peak_gbs(torch, dev):
    """Pinned host -> device copy bandwidth of this box (the roofline of the end-to-end leg)."""
    n = 1 << 30
    h = torch.empty(n, dtype=torch.uint8).pin_memory()
    d = torch.empty(n, dtype=torch.uint8, device=dev)
    best = 0.0
    d.copy_(h, non_blocking=True)          # first touch of both buffers
    torch.cuda.synchronize()
    for _ in range(8):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        d.copy_(h, non_blocking=True)
        e1.record()
        e1.synchronize()
        best = max(best, n / (e0.elapsed_time(e1) * 1e-3) / 1e9)
    return best


# ----------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from fastplong_b200 import synth_fast
    from fastplong_b200.binding import Engine

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    opt = workload_options(args.workload)
    opt.device = local
    wl_reads, wl_reps, mean_len, gen_kw, wl_desc = WORKLOADS[args.workload]
    tile_reads = args.reads or args.tile_reads or wl_reads
    replicas = args.replicas or wl_reps
    gen_kw = dict(gen_kw)
    if args.workload == "c3":
        gen_kw["planted"] = opt.adapter_fasta[:4]
    # ---- synthetic workload: DISTINCT reads generated on the device (torch Philox streams; the per-read structure is
    # drawn on the host).  Every rank draws the same read lengths and end pieces (equal work per GPU: weak scaling) and
    # its own bases and qualities. ----
    t0 = time.time()
    plan = synth_fast.read_plan(tile_reads, mean_len, SEED, **{k: v for k, v in gen_kw.items() if k in
                                                                ("p_polya", "planted", "p_planted", "min_len")})
    tile = synth_fast.ont_like_device(tile_reads, mean_len, SEED + 1000 * rank, dev, plan=plan,
                                      **{k: v for k, v in gen_kw.items() if k in ("q_mean", "q_sd", "q_clip")})
    torch.cuda.synchronize()
    gen_s = time.time() - t0
    tile_bytes = tile.n_bytes - 256            # drop the tail pad: replicas are laid back to back (multiple of 128)
    n_reads = tile_reads * replicas
    n_bases = tile.n_bases * replicas
    if replicas == 1:
        d_seq, d_qual = tile.seq, tile.qual
        offs = torch.from_numpy(tile.offsets).to(dev)
        lens = torch.from_numpy(tile.lens).to(dev)
    else:
        d_seq = torch.empty(tile_bytes * replicas + 256, dtype=torch.uint8, device=dev)
        d_qual = torch.empty_like(d_seq)
        for k in range(replicas):
            d_seq[k * tile_bytes:(k + 1) * tile_bytes].copy_(tile.seq[:tile_bytes])
            d_qual[k * tile_bytes:(k + 1) * tile_bytes].copy_(tile.qual[:tile_bytes])
        d_seq[tile_bytes * replicas:].zero_()
        d_qual[tile_bytes * replicas:].zero_()
        offs = (torch.from_numpy(tile.offsets).to(dev)[None, :] +
                (torch.arange(replicas, device=dev, dtype=torch.int64) * tile_bytes)[:, None]).reshape(-1).contiguous()
        lens = torch.from_numpy(tile.lens).to(dev).repeat(replicas).contiguous()
    torch.cuda.synchronize()

    # ---- config 2 says "auto-detected adapters": detect them on this input as the CLI's pre-pass would — the ten-mer tables
    # of Evaluator::evalAdapterAndReadNum on the device (fpl_eval_adapter_kmers), top key + extension on the host
    # (fpl_eval_pick_adapter, through fastplong_b200/evaluator.py), over the first <= 64 Ki reads / 512 Mbases; outside the timed path (SURVEY §8d) ----
    detected = None
    if args.workload == "c2" and not args.no_detect:
        from fastplong_b200 import evaluator, synth
        t0 = time.time()
        box = [None]
        if rank == 0:
            n_head = evaluator.evaluated_prefix(tile.lens)
            box[0] = evaluator.detect_adapters(tile.to_host(0, n_head), device=local)
        if world > 1:
            dist.broadcast_object_list(box, src=0)
        planted = (synth.ADAPTER_START, synth.ADAPTER_END)
        detected = {"start": box[0][0], "end": box[0][1], "equals_planted": tuple(box[0]) == planted,
                    "reads_evaluated": int(evaluator.evaluated_prefix(tile.lens)), "seconds": round(time.time() - t0, 2),
                    "how": "fpl_eval_adapter_kmers (device ten-mer tables) + fpl_eval_pick_adapter (getTopKey / extendKeyToAdapter "
                           "restated as host C++ in the C ABI), driven by fastplong_b200/evaluator.py with the reference's rules: "
                           "first <= 64 Ki reads / 512 Mbases of the input"}
        if box[0][0] != "auto":
            opt.start_adapter = box[0][0]
        if box[0][1] != "auto":
            opt.end_adapter = box[0][1]

    # ---- parity: the first reads of this very input, GPU library vs oracle, before anything is timed ----
    parity = None
    if not args.no_parity:
        csum = np.cumsum(tile.lens.astype(np.int64))
        n_par = int(min(tile_reads, max(16, np.searchsorted(csum, PARITY_BASES))))
        parity = parity_check(opt, tile.to_host(0, n_par))

    eng = Engine(opt)
    ext = torch.cuda.ExternalStream(eng.stream_ptr, device=dev)
    merge_cycles = 0
    if world > 1:
        # the C ABI's own communicator (ncclCommInitRank on rank 0's id); torch.distributed only carries the id
        ident = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            ident = torch.frombuffer(bytearray(Engine.comm_unique_id()), dtype=torch.uint8).to(dev)
        dist.broadcast(ident, 0)
        eng.comm_init(bytes(ident.cpu().numpy().tobytes()), rank, world)

    def step():
        eng.reset()
        eng.process_device(d_seq.data_ptr(), d_qual.data_ptr(), offs.data_ptr(), lens.data_ptr(), n_reads,
                           d_seq.numel())
        if world > 1:
            # Stats::merge / FilterResult::merge: one NCCL group on the library's stream, behind the kernels
            eng.allreduce_stats(merge_cycles)

    if world > 1:
        eng.reset()
        eng.process_device(d_seq.data_ptr(), d_qual.data_ptr(), offs.data_ptr(), lens.data_ptr(), n_reads, d_seq.numel())
        merge_cycles = eng.agree_cycles()      # once: every rank reduces the same [0, cycles) of every row
    for _ in range(max(args.warmup, 3)):
        step()
    eng.sync()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    # ---- timed region: K steps, device time by CUDA events on the library's stream ----
    eng.set_timing(True)
    l0 = eng.launch_count
    sampler = ClockSampler(physical_device_index(local))
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(ext)
    for _ in range(args.steps):
        step()
    ev1.record(ext)
    eng.sync()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    ms = ev0.elapsed_time(ev1)
    launches = eng.launch_count - l0
    ktimes = eng.kernel_times()
    eng.set_timing(False)
    dumped = dump_outputs(eng, n_reads, int(tile.lens.max()), args.dump_outputs) if args.dump_outputs and rank == 0 else None
    if world > 1:
        # every rank's clocks and step time: the value is the max over ranks, so a GPU that ran slower (power cap under an
        # 8-GPU load) shows here
        per_rank = [None] * world
        dist.all_gather_object(per_rank, {"rank": rank, "ms_per_step": round(ms / args.steps, 3), "sm_mhz": clocks["sm_mhz"],
                                          "reasons": clocks["reasons"]})
        clocks = dict(clocks, all_ranks=per_rank, min_sm_mhz=min((p["sm_mhz"] or 0) for p in per_rank),
                      reasons=sorted(set(r for p in per_rank for r in p["reasons"])))
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        tb = torch.tensor([float(n_bases)], device=dev, dtype=torch.float64)
        dist.all_reduce(tb)
        total_bases = float(tb.item())
    else:
        total_bases = float(n_bases)
    ms_per_step = ms / args.steps
    value = total_bases / (ms_per_step * 1e-3) / 1e9

    # ---- end to end through the C ABI with HOST buffers (pinned): H2D of the payload + D2H of the records ----
    # the per-GPU batch arrives as E2E_SUBMISSIONS host submissions; E2E_HOST_CHUNKS distinct chunks of this run's
    # input (1/64 of the reads each) are held in pinned memory and cycled
    from fastplong_b200 import PackedBatch
    from fastplong_b200.abi import RESULT_DTYPE
    e2e = None
    if not args.no_e2e:
        per = max(1, tile_reads // E2E_SUBMISSIONS)
        chunks = []
        for k in range(min(E2E_HOST_CHUNKS, max(1, tile_reads // per))):
            hb = tile.to_host(k * per, min(tile_reads, (k + 1) * per))
            pinned = [torch.from_numpy(x).pin_memory() for x in (hb.seq, hb.qual, hb.offsets, hb.lens)]
            res = torch.empty(hb.n_reads * RESULT_DTYPE.itemsize, dtype=torch.uint8).pin_memory()
            chunks.append((PackedBatch(*[x.numpy() for x in pinned]), res.numpy().view(RESULT_DTYPE), pinned, res))
        e2e_steps = max(1, min(args.steps, 3))
        sub_bases = sum(chunks[k % len(chunks)][0].n_bases for k in range(E2E_SUBMISSIONS))
        h2d = sum(2 * chunks[k % len(chunks)][0].n_bytes + 12 * chunks[k % len(chunks)][0].n_reads for k in range(E2E_SUBMISSIONS))
        d2h = sum(chunks[k % len(chunks)][0].n_reads for k in range(E2E_SUBMISSIONS)) * RESULT_DTYPE.itemsize

        def e2e_step():
            eng.reset()
            for k in range(E2E_SUBMISSIONS):
                hb, out = chunks[k % len(chunks)][:2]
                eng.process(hb, out=out)
            if world > 1:
                eng.allreduce_stats(merge_cycles)
                eng.sync()

        e2e_step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step()
        torch.cuda.synchronize()
        e2e_s = (time.perf_counter() - t0) / e2e_steps
        if world > 1:
            t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_s = float(t.item())
        pcie = h2d_peak_gbs(torch, dev) if world == 1 else None      # measured alone: with N ranks the links are shared
        e2e = {"value": round(sub_bases * world / e2e_s / 1e9, 3), "unit": "Gbases/s", "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "steps": e2e_steps,
               "how": "fpl_process_host on pinned host buffers, %d submissions/step (%d distinct chunks of this run's reads, "
                      "cycled); inside a call the upload runs in 16 MiB pieces on a copy stream and the kernels of a piece "
                      "start when it has arrived" % (E2E_SUBMISSIONS, len(chunks)),
               "achieved_pcie_gbs": round(h2d / e2e_s / 1e9, 2)}       # host -> device direction (the records go the other way)
        if pcie:
            ach = h2d / e2e_s / 1e9
            e2e["roofline"] = {"bound": "pcie h2d", "peak": round(pcie, 2), "unit": "GB/s", "achieved": round(ach, 2),
                               "frac": round(min(1.0, ach / pcie), 4),
                               "peak_source": "measured here: 1 GiB pinned host -> device copy, best of 8, CUDA events"}
            if ach > pcie:      # the copy measurement itself moves by a few % between runs of the same box
                e2e["roofline"]["note"] = "this leg ran faster than the copy measurement: at the peak (frac capped at 1)"

    # ---- roofline of the dominant kernel (largest share of the step's device time) ----
    peak, peak_src = peaks()
    alg_bytes_step = ALG_BYTES_PER_BASE * n_bases + ALG_BYTES_PER_READ * n_reads   # per GPU, per step
    kern = {}
    tot_kernel_ms = sum(v[0] for v in ktimes.values()) or 1.0
    for name, (kms, cnt) in ktimes.items():
        if cnt == 0:
            continue
        per_step_ms = kms / args.steps
        kern[name] = {"ms_per_step": round(per_step_ms, 4), "share": round(kms / tot_kernel_ms, 4),
                      "launches_per_step": cnt // args.steps,
                      "achieved_gbs": round(alg_bytes_step / (per_step_ms * 1e-3) / 1e9, 1) if per_step_ms > 0 else None}
    ours = {k: v for k, v in kern.items() if not k.startswith("nccl")}
    dom = max(ours, key=lambda k: ours[k]["ms_per_step"]) if ours else None
    traffic = None
    secondary = None      # SURVEY 8(d): the integer-pipe roofline, reported where it binds (from the committed ncu capture)
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if dom and os.path.exists(tp):
        try:
            tj = json.load(open(tp))
            if dom in tj:   # DRAM bytes per algorithmic byte from the committed ncu --set full capture
                nl = max(1, kern[dom]["launches_per_step"])
                traffic = tj[dom]["dram_bytes_per_alg_byte"] * alg_bytes_step / nl
                if "alu_pipe_active_pct" in tj[dom]:
                    secondary = {"bound": "integer logic pipe (LOP3/SHF/PRMT issue slots)",
                                 "frac": round(tj[dom]["alu_pipe_active_pct"] / 100.0, 4),
                                 "fma_pipe_frac": round(tj[dom].get("fma_pipe_active_pct", 0) / 100.0, 4),
                                 "source": tj[dom].get("source", "ncu --set full capture under profiles/ (not measured live)")}
        except Exception:
            traffic = None
            secondary = None
    roofline = None
    if dom:
        nl = max(1, kern[dom]["launches_per_step"])
        achieved = kern[dom]["achieved_gbs"]
        roofline = {"kernel": dom, "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": round(achieved / peak, 4), "traffic": traffic, "peak_source": peak_src,
                    "alg_bytes_per_launch": alg_bytes_step / nl, "avg_launch_ms": round(kern[dom]["ms_per_step"] / nl, 5),
                    "launches_per_step": nl, "secondary": secondary,
                    "whole_path": {"achieved": round(alg_bytes_step / (ms_per_step * 1e-3) / 1e9, 1),
                                   "frac": round(alg_bytes_step / (ms_per_step * 1e-3) / 1e9 / peak, 4),
                                   "note": "one pass of algorithmic bytes over the whole step (the path makes several passes)"}}
        if "k_scan" in kern and dom != "k_scan":
            a = kern["k_scan"]["achieved_gbs"]
            roofline["adapter_quality_kernel"] = {"kernel": "k_scan", "achieved": a, "frac": round(a / peak, 4),
                                                  "avg_launch_ms": kern["k_scan"]["ms_per_step"]}

    # ---- parity at full size (single-GPU runs; after everything that is timed): one more device-resident pass of the whole
    # batch, then its records / Stats blocks / counters are checked (full_scale_check).  Multi-GPU runs process the same
    # kind of batch per rank with the same kernels and skip it (their ranks would idle at the barrier meanwhile). ----
    full = None
    if world == 1 and parity is not None and not args.no_full_check:
        try:
            eng.reset()
            eng.process_device(d_seq.data_ptr(), d_qual.data_ptr(), offs.data_ptr(), lens.data_ptr(), n_reads, d_seq.numel())
            eng.sync()
            full = full_scale_check(torch, eng, opt, tile, d_seq, d_qual, offs.cpu().numpy(), lens.cpu().numpy(), tile_reads,
                                    mean_len)
        except AssertionError as e:
            full = {"ok": False, "error": str(e)[:500]}
        except Exception as e:      # the checker itself failed (time budget, memory): reported, never fatal for the line
            full = {"ok": None, "error": "%s: %s" % (type(e).__name__, str(e)[:400])}
        torch.cuda.empty_cache()

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_baseline = reference_cpu_run(sample_reads=REF_SAMPLE_READS, repeats=1)

    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    line = {
        "metric": "Gbases/s processed (adapter-trim + Q-filter + pre/post stats)", "value": round(value, 3),
        "unit": "Gbases/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": round(ms_per_step, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": wl_desc,
                   "reads_per_gpu": n_reads, "bases_per_gpu": n_bases, "mean_len": mean_len,
                   "input": (f"{tile_reads} distinct reads generated on the device (fastplong_b200/synth_fast.py, seeded; torch "
                             "Philox streams for bases and qualities)" +
                             (f", replicated {replicas}x in HBM" if replicas > 1 else "")),
                   "adapters": detected if detected else "planted strings given as -s / -e",
                   "l2": "inputs (2 x %.1f GB) larger than L2; no flush needed" % (d_seq.numel() / 1e9),
                   "parallelism": f"reads sharded over {world} GPU(s), equal bases per GPU; Stats/FilterResult merged by one NCCL "
                                  "all-reduce group per step issued by the C ABI (fpl_allreduce_stats) on the library's stream"
                   if world > 1 else "single GPU", "read_tiling": (os.environ.get("FPL_TILE_MBASES") + " Mbases") if os.environ.get("FPL_TILE_MBASES") else "none (every kernel streams the whole batch)",
                   "input_gen_s": round(gen_s, 1),
                   "variants": {"k_scan_jit": "v1 (round 1)" if os.environ.get("FPL_JIT_V1") else "v2",
                                "k_cycle_stats_staging": "1-D TMA (cp.async.bulk + mbarrier)" if os.environ.get("FPL_CS_TMA", "0") not in ("", "0")
                                else "cp.async (LDGSTS) ring"}},
        "parity_checked": parity is not None, "parity": parity, "parity_full_scale": full,
        "clocks": clocks,
        "e2e": e2e,
        "gpu_launches": int(launches),
        "collective_ms": kern.get("nccl_allreduce(stats)", {}).get("ms_per_step") if world > 1 else None,
        "roofline": roofline, "kernels": kern, "cpu_baseline": cpu_baseline,
    }
    if dumped:
        line["dumped_outputs"] = dumped
    emit(line)


# ----------------------------------------------------------------------------------------------------------------
_SAMPLE_CACHE = {}


def reference_cpu_run(sample_reads, repeats):
    """fastplong_ref (the unmodified reference, oracle/_ref) on a bounded sample of the same workload, plain FASTQ
    on tmpfs, all the worker threads it accepts (-w min(16, nproc)).  Returns the cpu_baseline object."""
    from fastplong_b200 import synth
    binary = os.path.join(ROOT, "oracle", "_ref", "fastplong_ref")
    if not os.path.exists(binary):
        return {"value": None, "unit": "Gbases/s", "cores": 0, "kind": "reference",
                "sample": "oracle/_ref/fastplong_ref not built"}
    tmp = "/dev/shm" if os.path.isdir("/dev/shm") else "/tmp"
    fq = os.path.join(tmp, f"fpl_bench_{os.getpid()}_{sample_reads}.fq")
    if fq in _SAMPLE_CACHE:
        n_bases = _SAMPLE_CACHE[fq]
    else:
        from fastplong_b200 import synth_fast
        batch = synth_fast.ont_like_fast(sample_reads, MEAN_LEN, SEED)      # the generator of the GPU arm, on the CPU
        synth.to_fastq(batch, fq)
        n_bases = _SAMPLE_CACHE[fq] = batch.n_bases
        import atexit
        atexit.register(lambda: os.path.exists(fq) and os.remove(fq))
    cores = min(16, os.cpu_count() or 1)
    opt = workload_options()
    opt.start_adapter = opt.end_adapter = "auto"   # the binary runs its own detection pre-pass
    best = None
    try:
        for _ in range(repeats):
            cmd = [binary, "-i", fq, "-o", fq + ".out", "-j", fq + ".json", "-h", fq + ".html", "-w", str(cores), "-V"]
            cmd += opt.cli_flags()
            # -V makes the reference log "start to load data" (src/seprocessor.cpp:334) and "start to generate reports"
            # (:105-106); its own timestamps have 1 s resolution, so the lines are stamped here as they arrive
            t0 = time.perf_counter()
            pr = subprocess.Popen(cmd, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, text=True, bufsize=1)
            t_load = t_rep = None
            tail = []
            for ln in pr.stderr:
                now = time.perf_counter()
                tail.append(ln)
                if t_load is None and "start to load data" in ln:
                    t_load = now
                elif "start to generate reports" in ln:
                    t_rep = now
            pr.wait()
            wall = time.perf_counter() - t0
            if pr.returncode != 0:
                return {"value": None, "unit": "Gbases/s", "cores": cores, "kind": "reference",
                        "sample": "fastplong_ref failed: " + "".join(tail)[-200:]}
            phase = (t_rep - t_load) if (t_load is not None and t_rep is not None and t_rep > t_load) else wall
            if best is None or phase < best[0]:
                best = (phase, wall)
    finally:
        for suffix in (".out", ".json", ".html"):
            try:
                os.remove(fq + suffix)
            except OSError:
                pass
    phase, wall = best
    return {"value": round(n_bases / phase / 1e9, 5), "unit": "Gbases/s", "cores": cores, "kind": "reference",
            "sample": f"{sample_reads} reads / {n_bases} bases of the same generator, fastplong_ref -w {cores}, plain FASTQ on "
                      f"tmpfs; value = bases / processing phase ({phase:.2f} s between the -V lines 'start to load data' and "
                      f"'start to generate reports': reader + workers + writer, the path itself); the whole binary took "
                      f"{wall:.2f} s (adapter detection pre-pass, Stats allocation and JSON/HTML reports included)",
            "phase_s": round(phase, 3), "wall_s": round(wall, 3), "whole_binary_gbases_s": round(n_bases / wall / 1e9, 5),
            "bases": n_bases}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample_reads = REF_SAMPLE_READS
    for _ in range(max(args.warmup, 1)):
        reference_cpu_run(sample_reads, 1)
    walls, base = [], None
    for _ in range(args.steps):
        base = reference_cpu_run(sample_reads, 1)
        if base["value"] is None:
            emit({"impl": "reference", "unavailable": base["sample"]})
            return
        walls.append(base["phase_s"])
    ms = 1e3 * sum(walls) / len(walls)      # a step = the processing phase of one run over the sample
    value = base["bases"] / (ms * 1e-3) / 1e9
    cb = dict(base)
    cb["value"] = round(value, 5)
    line = {"impl": "reference", "metric": "Gbases/s processed (adapter-trim + Q-filter + pre/post stats)",
            "value": round(value, 5), "unit": "Gbases/s", "n_gpus": int(os.environ.get("WORLD_SIZE", "1")),
            "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": round(ms, 2), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": "configs[1] shape, bounded sample: %d ONT reads mean 15 kb (%.1f Gbases) per step, auto-detected "
                                   "adapters + --cut_front --cut_tail -W 10 (reference CPU build, host cores only; a step is timed "
                                   "over the binary's processing phase)" % (sample_reads, base["bases"] / 1e9)},
            "cpu_baseline": cb,
            "e2e": {"value": round(value, 5), "unit": "Gbases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


_JSON_OUT = None


def claim_stdout():
    """stdout carries exactly one JSON line.  Libraries write there too (NCCL prints its version banner with a plain
    printf when NCCL_DEBUG=VERSION): keep a private handle on the real stdout for the line and point file descriptor 1
    at stderr for everybody else."""
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line):
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS),
                    help="c2 = BASELINE configs[1] (the bench line); the others = the remaining BASELINE config shapes")
    ap.add_argument("--reads", type=int, default=0, help="distinct reads per GPU (default: the workload's)")
    ap.add_argument("--tile-reads", type=int, default=0, help="alias of --reads (profiling: a small tile ...)")
    ap.add_argument("--replicas", type=int, default=0, help="... replicated this many times in HBM")
    ap.add_argument("--no-detect", action="store_true", help="profiling aid: skip the adapter auto-detection pre-pass (use the planted strings)")
    ap.add_argument("--no-parity", action="store_true", help="profiling aid: skip the oracle comparison of the first reads")
    ap.add_argument("--no-full-check", action="store_true", help="profiling aid: skip the full-size parity check behind the timed legs")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="profiling aid: skip the end-to-end leg (keeps an ncu launch list short)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (Stats blocks, counters, sampled records)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
