#!/usr/bin/env python
"""bench.py -- headline benchmark of the SPEV-TTS spectral hot path on B200.

    python bench.py --gpus N --steps K --warmup W            (our arm: sm_100a kernels)
    python bench.py --impl reference --gpus N --steps K ...  (reference arm: CPU path)

Metric (BASELINE.json): mel frames/s (STFT -> 80-mel log-spectrogram) on the LJSpeech-shaped cache build
(configs[3]: 13,100 synthetic utterances of 1-10 s at 22.05 kHz = 6.35 GB of float32 samples, ~6.2 M frames -- far
larger than the 126 MB L2, so no L2 flush is needed between steps).

STRONG scaling, as configs[3] says: the corpus is FIXED (seed 4, the same 13,100 utterances for every N) and is
sharded by utterance across the N ranks (greedy length balancing); one "step" is the whole multi-GPU job -- every
rank's fused kernel over its shard AND the NCCL gather of the shards into rank 0's cache (chunked, overlapped with the
kernel).  `value` = corpus frames / that time; `kernel_only` (no gather: every data-parallel rank keeps its shard
resident), `gather_serial` (kernel, then gather) and the gather's own bandwidth are reported beside it.  At N = 1
there is nothing to gather and a step is one launch over the whole corpus.

The same JSON line also carries the second half of the metric, Griffin-Lim audio-seconds/s on configs[2] (16 x
[80,800] log-mels, 60 iterations), with its own roofline, under "griffinlim", and the LengthRegulator / bucketize
timing on configs[1] under "length_regulator".

The reference arm times the reference's own CPU implementation of the path: real librosa when it is importable on the
box, else the oracle restatement of librosa 0.11 (``oracle/librosa_restated.py``; see DESIGN.md), fanned over all host
cores, on a bounded sample of the same workload.  Its `value` and `ms_per_step` share one basis: wall time of the
pooled map over the sample.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SR, HOP, N_MELS = 22050, 256, 80
ALG_BYTES_PER_FRAME = 1344          # 256 new samples * 4 B read + 80 * 4 B written (SURVEY 8d)
NCU_DRAM_BYTES_PER_FRAME = 1320.2   # (dram__bytes_read + dram__bytes_write) of k_stft_mel<0,5> / frames, profiles/r02_ncu_k_stft_mel.txt
NCU_TRAFFIC_SOURCE = ("ncu --set full, profiles/r02_ncu_k_stft_mel.txt: 736.7 MB read + 212.6 MB written for 719,053 frames "
                      "= 1,320 B/frame (below the 1,344 algorithmic bytes: rows of neighbouring tiles share DRAM sectors)")
NCU_ISSUE_NOTE = {"warp_instr_per_frame": 1042, "issue_active_pct": 65.2, "lsu_wavefront_pct": 61.4, "fma_pipe_pct": 40.8,
                  "note": "co-limited by issue slots and the shared-memory pipe, not HBM"}
GL_BYTES_PER_FRAME_ITER = 20516     # SURVEY 8d
N_UTTS = 13100


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


# ----------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ts, line in self.rows:
            if t0 is not None and not (t0 - 0.05 <= ts <= t1 + 0.15):
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------
# CPU reference path (oracle), fanned over host cores
# ----------------------------------------------------------------------------------------------
def _cpu_worker_init():
    """one BLAS/OpenMP thread per worker process (the pool supplies the parallelism)"""
    try:
        from threadpoolctl import threadpool_limits
        globals()["_tp_limit"] = threadpool_limits(1)
    except Exception:
        pass


_CPU_WAVES = None          # the bounded sample, generated in the parent before the pool forks
_USE_LIBROSA = False


def have_librosa() -> bool:
    try:
        import librosa  # noqa: F401
        import librosa.feature  # noqa: F401
        return hasattr(librosa.feature, "melspectrogram")
    except Exception:
        return False


def _cpu_logmel_job(i):
    y = _CPU_WAVES[i]
    if _USE_LIBROSA:       # the reference's own statements, spev_real_metrics.py:363-367 + :421
        import librosa
        mel = librosa.feature.melspectrogram(y=y, sr=SR, n_fft=1024, hop_length=HOP, n_mels=N_MELS)
        mel = np.clip(np.log(np.clip(mel, 1e-5, None)), -10, 2)
        m = np.ascontiguousarray(mel.T, dtype=np.float32)
    else:
        from oracle import librosa_restated as lr
        m = lr.reference_logmel(y)
    return m.shape[0]


def _cpu_gl_job(args):
    seed, T, n_iter = args
    from oracle import librosa_restated as lr
    rng = np.random.default_rng(seed)
    lm = np.clip(-4 + 2 * rng.standard_normal((80, T)), -10, 2).astype(np.float32)
    t = time.perf_counter()
    lr.reference_vocoder_infer(lm, n_iter=n_iter, seed=seed, lbfgs=True)
    return (T - 1) * HOP / SR, time.perf_counter() - t


class CpuLogmel:
    """The reference's CPU log-mel path on a bounded sample of the cfg4 corpus, one utterance per task over a pool of
    `procs` single-threaded workers.  One time basis everywhere: WALL time of the pooled map (pool start-up and data
    generation happen once, before the first step)."""

    def __init__(self, n_utts: int, procs: int, seed: int = 4):
        import multiprocessing as mp
        from tests import synth
        global _CPU_WAVES, _USE_LIBROSA
        lens = synth.utterance_lengths(seed=seed, n_utts=N_UTTS)[:n_utts]
        rng = np.random.default_rng(seed)
        _CPU_WAVES = [(0.05 * rng.standard_normal(int(n))).astype(np.float32) for n in lens]
        _USE_LIBROSA = have_librosa()
        self.kind = "reference" if _USE_LIBROSA else "port"
        self.impl = "librosa.feature.melspectrogram + log/clip" if _USE_LIBROSA else "oracle/librosa_restated.py"
        self.n, self.procs = len(lens), procs
        os.environ.setdefault("OMP_NUM_THREADS", "1")
        self.pool = mp.get_context("fork").Pool(procs, initializer=_cpu_worker_init) if procs > 1 else None

    def step(self):
        """-> (frames/s, frames, wall seconds)"""
        t = time.perf_counter()
        if self.pool is not None:
            res = self.pool.map(_cpu_logmel_job, range(self.n), chunksize=4)
        else:
            res = [_cpu_logmel_job(i) for i in range(self.n)]
        wall = time.perf_counter() - t
        frames = int(sum(res))
        return frames / wall, frames, wall

    def close(self):
        if self.pool is not None:
            self.pool.close()
            self.pool.join()


def _cpu_pyin_job(args):
    seed, n = args
    from oracle import pyin_restated as po
    from tests import synth
    y = synth.voiced_unvoiced(seed=seed, n=n)[0]
    t = time.perf_counter()
    f0, _, _ = po.pyin(y)
    return len(f0), n / SR, time.perf_counter() - t


def cpu_pyin_throughput(n_utts: int, procs: int, seed: int = 4):
    """frames/s and audio-s/s of the restated librosa.pyin on cfg4-shaped utterances."""
    import multiprocessing as mp
    from tests import synth
    lens = synth.utterance_lengths(seed=seed, n_utts=N_UTTS)[:n_utts]
    jobs = [(i % 16, int(n)) for i, n in enumerate(lens)]
    t = time.perf_counter()
    if procs > 1:
        with mp.get_context("fork").Pool(min(procs, n_utts), initializer=_cpu_worker_init) as pool:
            res = pool.map(_cpu_pyin_job, jobs)
    else:
        res = [_cpu_pyin_job(j) for j in jobs]
    wall = time.perf_counter() - t
    busy = sum(r[2] for r in res) / max(1, min(procs, n_utts))
    return sum(r[0] for r in res) / busy, sum(r[1] for r in res) / busy, wall


def cpu_gl_throughput(n_items: int, T: int, n_iter: int, procs: int):
    import multiprocessing as mp
    jobs = [(300 + i, T, n_iter) for i in range(n_items)]
    t = time.perf_counter()
    if procs > 1:
        with mp.get_context("fork").Pool(min(procs, n_items), initializer=_cpu_worker_init) as pool:
            res = pool.map(_cpu_gl_job, jobs)
    else:
        res = [_cpu_gl_job(j) for j in jobs]
    wall = time.perf_counter() - t
    return sum(r[0] for r in res) / wall, wall


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    n_utts = args.ref_utts
    cpu = CpuLogmel(n_utts, cores)
    for _ in range(args.warmup):
        cpu.step()
    walls, frames = [], 0
    for _ in range(args.steps):
        _, frames, wall = cpu.step()
        walls.append(wall)
    cpu.close()
    ms = float(np.mean(walls)) * 1e3
    value = frames / (ms * 1e-3)                      # same basis as ms_per_step: wall time of one pooled pass
    gl_v, gl_wall = cpu_gl_throughput(min(cores, 16), 800, 60, cores)
    sample = f"{n_utts} of {N_UTTS} cfg4 utterances per step ({frames} frames), {cores} processes, {cpu.impl}"
    line = {
        "impl": "reference", "metric": "mel frames/s (STFT->80-mel log, cache build)", "value": value,
        "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64 FFT / f32 mel (librosa semantics)", "data": "synthetic",
        "config": {"workload": "cfg4: 13,100 synthetic utterances 1-10 s @22.05 kHz (bounded sample)",
                   "n_fft": 1024, "hop": 256, "n_mels": 80},
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": cores, "kind": cpu.kind, "sample": sample,
                         "time_basis": "wall time of the pooled map"},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "griffinlim": {"value": gl_v, "unit": "audio-s/s", "n_iter": 60, "cores": cores,
                       "sample": f"{min(cores, 16)} x [80,800], wall {gl_wall:.1f}s, NNLS L-BFGS-B on",
                       "time_basis": "wall time of the pooled map"},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ----------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    import spev_tts_b200 as sp
    from spev_tts_b200 import cache as spcache
    from tests import synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py (our arm) needs a B200; there is no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = spcache.bind_to_gpu_numa_node(dev) if world > 1 else {"bound": False}   # before any pinned allocation
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    sp.load()
    hbm_peak, peak_src = peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---------------- cfg4: the FIXED 13,100-utterance corpus, sharded by utterance over the ranks --------
    lens = synth.utterance_lengths(seed=4, n_utts=args.utts)
    plan = spcache.plan_shards(lens, world, n_chunks=args.chunks)
    bld = spcache.ShardedCacheBuilder(plan, rank, dev, dst=0, sr=SR, n_mels=N_MELS, reserve_sms=args.reserve_sms)
    ctx = bld.ctx
    mine = plan.shards[rank]
    starts = bld.sample_off                     # item starts are multiples of 4 samples (16-B cp.async path)
    total = int(starts[-1])
    # every rank derives the same corpus from seed 4 and keeps its shard's utterances (setup, untimed)
    full_starts = spcache.aligned_offsets(lens)
    g = torch.Generator(device=dev).manual_seed(4)
    full = torch.empty(int(full_starts[-1]), dtype=torch.float32, device=dev)
    blk = 1 << 27
    for s0 in range(0, full.numel(), blk):       # generate in blocks to bound the temporary
        e0 = min(full.numel(), s0 + blk)
        full[s0:e0] = torch.randn(e0 - s0, generator=g, device=dev) * 0.05
    if world == 1:
        samples = full
    else:
        samples = torch.zeros(total, dtype=torch.float32, device=dev)
        spcache.copy_segments(full.view(-1, 1), samples.view(-1, 1), full_starts[mine], starts[:-1], lens[mine])
        torch.cuda.synchronize(dev)
    del full
    torch.cuda.empty_cache()
    batch = bld.batch_all
    F = batch.n_frames                           # this rank's frames
    F_total = plan.n_rows                        # corpus frames (the same for every N)
    out = bld.alloc_out()                        # rank 0: the gathered cache [F_total, 80]; others: their shard
    out_local = bld.local_rows(out)

    def timed(fn, n, warm):
        """n steps back to back, bracketed by barrier + synchronize; -> (max-over-ranks ms per step, this rank's
        mean per-step ms from CUDA events around each step)"""
        for _ in range(warm):
            fn()
        barrier()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
        a0 = torch.cuda.Event(enable_timing=True); a1 = torch.cuda.Event(enable_timing=True)
        barrier()
        a0.record()
        for ea, eb in evs:
            ea.record(); fn(); eb.record()
        a1.record()
        barrier()
        return max_over_ranks(a0.elapsed_time(a1)) / n, float(np.mean([ea.elapsed_time(eb) for ea, eb in evs]))

    W = max(args.warmup, 3)
    sampler = ClockSampler(local).start() if rank == 0 else None
    time.sleep(0.3)
    t0 = time.perf_counter()
    # (1) kernels only: every rank builds its shard and keeps it (the sharded-resident alternative)
    ko_ms, kern_ms = timed(lambda: bld.build(samples, out, gather=False), args.steps, W)
    kern_ms_max = max_over_ranks(kern_ms)
    launches_per_step = 1
    gather = None
    bld_p = out_p = None
    if world == 1:
        ms_per_step = ko_ms
    else:
        # (2) the whole job: kernels + gather into rank 0, chunked and overlapped  -> the headline value
        l0 = bld.launches
        ov_ms, _ = timed(lambda: bld.build(samples, out, gather=True, overlap=True), args.steps, W)
        launches_per_step = (bld.launches - l0) // (args.steps + W)
        # (3) for comparison: kernel, then one grouped gather (no overlap), and the gather alone
        se_ms, _ = timed(lambda: bld.build(samples, out, gather=True, overlap=False), max(3, args.steps // 2), 1)
        peers_rows = F_total - int(plan.row_off[1] - plan.row_off[0])
        nbytes = peers_rows * N_MELS * 4
        gather = {"bytes_into_root": nbytes,
                  "nccl": {"backend": "ncclSend/ncclRecv (batch_isend_irecv), receives land in their final rows",
                           "overlapped_ms_per_step": ov_ms, "serial_ms_per_step": se_ms,
                           "gather_alone_ms": se_ms - ko_ms,
                           "gather_alone_GBps": nbytes / max(1e-9, (se_ms - ko_ms) * 1e-3) / 1e9,
                           "reserved_sms": args.reserve_sms,
                           "note": "NCCL's send/recv kernels need SMs; the FFT CTAs each fill one, so the kernels run "
                                   "on 148 - reserved SMs while a transfer is in flight"},
                  "kernel_only_ms_per_step": ko_ms, "chunks_per_rank": args.chunks,
                  "limiter": "root NVLink ingress: (N-1)/N of the 1.99 GB cache must enter rank 0; lower bound = bytes / "
                             "measured peer-copy bandwidth (770 GB/s per direction, B200_PROFILING.md)",
                  "ingress_floor_ms": nbytes / 770e9 * 1e3}
        ms_per_step, transport = ov_ms, "nccl"
        bld_p = out_p = None
        if args.transport in ("best", "p2p"):
            try:
                bld_p = spcache.ShardedCacheBuilder(plan, rank, dev, dst=0, sr=SR, n_mels=N_MELS, transport="p2p")
                out_p = bld_p.alloc_out()
                l0 = bld_p.launches
                pv_ms, _ = timed(lambda: bld_p.build(samples, out_p, gather=True, overlap=True), args.steps, W)
                p_launches = (bld_p.launches - l0) // (args.steps + W)
                ps_ms, _ = timed(lambda: bld_p.build(samples, out_p, gather=True, overlap=False), max(3, args.steps // 2), 1)
                gather["p2p"] = {"backend": "copy-engine pushes into the root's symmetric-memory window (cudaMemcpyAsync over "
                                            "NVLink, no SMs), signal-pad barrier",
                                 "overlapped_ms_per_step": pv_ms, "serial_ms_per_step": ps_ms,
                                 "gather_alone_ms": ps_ms - ko_ms,
                                 "gather_alone_GBps": nbytes / max(1e-9, (ps_ms - ko_ms) * 1e-3) / 1e9}
                if pv_ms < ms_per_step or args.transport == "p2p":
                    ms_per_step, transport, launches_per_step = pv_ms, "p2p", p_launches
            except RuntimeError as e:
                gather["p2p"] = {"unavailable": str(e)[:300]}
                bld_p = out_p = None
        gather["headline_transport"] = transport
    t1 = time.perf_counter()
    if args.dump_outputs and rank == 0:
        headline_out = out_p if gather is not None and gather["headline_transport"] == "p2p" else out
        dump_cache_sample(args.dump_outputs, headline_out, plan)
    value = F_total / (ms_per_step * 1e-3)
    kernel_only = {"value": F_total / (ko_ms * 1e-3), "unit": "frames/s", "ms_per_step": ko_ms,
                   "note": "no gather: each data-parallel rank keeps its shard resident (ResidentCache)"}
    achieved = ALG_BYTES_PER_FRAME * F / (kern_ms * 1e-3) / 1e9      # GB/s, this rank's kernel
    # ---------------- e2e: pinned host samples -> public API -> pinned host cache (this rank's shard) -------
    e2e = None
    if not args.no_e2e:
        host = torch.empty(total, dtype=torch.float32).pin_memory()
        host.copy_(samples)
        out_host = torch.empty((F, N_MELS), dtype=torch.float32).pin_memory()
        # PCIe denominators: rank 0 alone first (the others wait), then every rank at once -- the host side (root
        # complexes, memory controllers) is shared, and that, not a kernel, is what limits e2e as ranks are added
        pcie = None
        if world > 1:
            barrier()
            if rank == 0:
                pcie = measure_pcie(dev, host, out_host)
            barrier()
        together = measure_pcie(dev, host, out_host)
        if world == 1:
            pcie = together
        else:
            agg = sum_over_ranks((total * 4 + F * N_MELS * 4) / 1e9) / max_over_ranks((total * 4 + F * N_MELS * 4) / 1e9 / together["duplex_GBps"])
            if rank == 0:
                pcie["all_ranks_at_once"] = {"rank0": together, "aggregate_duplex_GBps": agg,
                                             "note": "every rank copying its shard in both directions at the same time"}
            else:
                pcie = together
        builder = spcache.LogMelCacheBuilder(dev, sr=SR, n_mels=N_MELS)
        cplan = spcache.plan_chunks(lens[mine], builder.chunk_samples, starts)
        for _ in range(2):                                                    # warm-up (allocs, descriptors; the first build
            builder.build(host, lens[mine], out_host=out_host, plan=cplan)    # after them still runs ~15 % slow: see ms_per_step_all)
        torch.cuda.synchronize(dev)
        n_e2e = max(1, min(args.steps, args.e2e_steps))
        barrier()
        # every step is timed on its own (event after each build) and the MEDIAN step is reported, all steps listed: the
        # host side of this pool is shared and a build now and then runs 30-50 % slower than its neighbours in the same
        # process (same buffers, same code) -- the mean of three steps was a lottery (125 ... 187 ms across runs)
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(n_e2e + 1)]
        l0 = builder.launches
        evs[0].record()
        for i in range(n_e2e):
            builder.build(host, lens[mine], out_host=out_host, plan=cplan)
            evs[i + 1].record()
        barrier()
        e2e_steps_ms = [max_over_ranks(evs[i].elapsed_time(evs[i + 1])) for i in range(n_e2e)]
        e2e_ms = float(np.median(e2e_steps_ms))
        e2e_launches = (builder.launches - l0) // n_e2e
        ok = bool(torch.equal(out_host[: 4096].to(dev), out_local[: 4096]))
        h2d_b, d2h_b = total * 4, F * N_MELS * 4
        floor_ms = max(h2d_b / pcie["h2d_GBps"], d2h_b / pcie["d2h_GBps"]) / 1e6
        e2e = {"value": F_total / (e2e_ms * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": h2d_b,
               "d2h_bytes_per_step": d2h_b, "ms_per_step": e2e_ms, "steps": n_e2e,
               "statistic": "median step (max over ranks per step)", "ms_per_step_all": e2e_steps_ms,
               "launches_per_step": e2e_launches, "matches_device_result": ok,
               "api": "spev_tts_b200.cache.LogMelCacheBuilder.build (pinned host in/out, 3-stream pipeline)",
               "bytes_note": "per rank (its shard); all ranks copy concurrently",
               "roofline": {"bound": "pcie", "peak": pcie, "floor_ms": floor_ms, "frac": floor_ms / e2e_ms,
                            "duplex_floor_ms": (h2d_b + d2h_b) / pcie["duplex_GBps"] / 1e6,
                            "frac_of_duplex_floor": (h2d_b + d2h_b) / pcie["duplex_GBps"] / 1e6 / e2e_ms,
                            "note": "floor = max(H2D bytes / measured pinned H2D GB/s, D2H bytes / measured D2H GB/s) "
                                    "of rank 0 measured ALONE in this run (PCIe is full duplex); duplex_floor = all bytes / "
                                    "the rate measured with both directions copying at once (what the pipelined build "
                                    "actually faces: the two directions share the host side); at N > 1 compare with "
                                    "all_ranks_at_once: the shared host side is the limiter"},
               "host_numa_binding_rank0": numa}
        # extra: the same corpus as 16-bit PCM on the host (the on-disk format of LJSpeech-style
        # corpora; pcm/32768 is exactly what the reference's loader produces) -> half the H2D bytes
        pcm = (samples.clamp(-1, 1) * 32767).to(torch.int16)
        del host                                      # one big pinned input buffer at a time
        host16 = torch.empty(total, dtype=torch.int16).pin_memory()
        host16.copy_(pcm)
        del pcm
        builder.build(host16, lens[mine], out_host=out_host, plan=cplan)
        torch.cuda.synchronize(dev)
        barrier()
        pevs = [torch.cuda.Event(enable_timing=True) for _ in range(n_e2e + 1)]
        pevs[0].record()
        for i in range(n_e2e):
            builder.build(host16, lens[mine], out_host=out_host, plan=cplan)
            pevs[i + 1].record()
        barrier()
        pcm_ms = float(np.median([max_over_ranks(pevs[i].elapsed_time(pevs[i + 1])) for i in range(n_e2e)]))
        pfloor = max(total * 2 / pcie["h2d_GBps"], d2h_b / pcie["d2h_GBps"]) / 1e6
        e2e["pcm16_host_input"] = {"value": F_total / (pcm_ms * 1e-3), "unit": "frames/s", "ms_per_step": pcm_ms,
                                   "h2d_bytes_per_step": total * 2, "d2h_bytes_per_step": d2h_b,
                                   "roofline_frac_of_pcie_floor": pfloor / pcm_ms,
                                   "note": "input quantised to int16 (not the float32 arm's exact values)"}
        del host16, out_host, builder
    clocks = sampler.stop(t0, t1) if sampler else None

    # ---------------- gather integrity: every rank's rows arrived where the plan says (exact checksums) ---------
    if world > 1:
        for name, b_, o_ in (("nccl", bld, out), ("p2p", bld_p, out_p)):
            if b_ is None:
                continue
            if rank == 0:
                o_.fill_(-1.0)
            b_.build(samples, o_, gather=True, overlap=True)
            mysum = b_.local_rows(o_).double().sum().reshape(1)
            sums = [torch.zeros_like(mysum) for _ in range(world)]
            dist.all_gather(sums, mysum)
            if rank == 0:
                gather[name]["rows_checksum_matches_every_rank"] = all(
                    bool(o_[int(plan.row_off[r]): int(plan.row_off[r + 1])].double().sum() == sums[r][0]) for r in range(world))
        del out_p, bld_p

    # ---------------- second half of the metric and the other configs ------------------------------------------
    gl = lr_res = tc = cfg5 = feat = coll = pyin_res = None
    lens_mine = lens[mine]
    if not args.no_gl:
        cfg5 = bench_cfg5(sp, dev, hbm_peak, spcache, world, max_over_ranks, sum_over_ranks)     # all ranks (aggregated)
        if rank == 0:
            pyin_res = bench_pyin(sp, dev, hbm_peak, args, world == 1 and not args.no_cpu)
            tc = bench_mel_gemm_tc(sp, dev, samples, lens_mine, starts, hbm_peak, out_local)
            feat = bench_frame_features(sp, dev, samples, lens_mine, starts, hbm_peak)
            coll = bench_collate(sp, dev, out_local, batch, hbm_peak)
            gl = bench_griffinlim(sp, dev, hbm_peak, args)
            lr_res = bench_length_regulator(sp, dev, args)
    parity = None
    if rank == 0 and not args.no_cpu:
        # spot-check of the measured result against the CPU oracle on the same inputs (checker only)
        from oracle import librosa_restated as lr_oracle
        errs = []
        nl = len(mine)
        for i in (0, 1, nl // 2, nl - 1):
            yy = samples[int(starts[i]): int(starts[i]) + int(lens_mine[i])].cpu().numpy()
            ref_lm = lr_oracle.reference_logmel(yy)
            got_lm = out_local[int(batch.frame_off[i]): int(batch.frame_off[i + 1])].cpu().numpy()
            errs.append(float(np.abs(ref_lm - got_lm).max()))
        parity = {"logmel_max_abs_err_vs_oracle": max(errs), "tolerance": 1e-4, "utterances_checked": 4}
        if not args.no_gl:
            parity.update(parity_griffinlim(sp, dev, lr_oracle))
    del samples, out, out_local
    torch.cuda.empty_cache()
    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu:
            cores = os.cpu_count() or 1
            c = CpuLogmel(args.ref_utts, cores)
            c.step()                                                  # warm-up: worker imports, page faults
            v, frames, wall = c.step()
            c.close()
            cpu = {"value": v, "unit": "frames/s", "cores": cores, "kind": c.kind,
                   "sample": f"{args.ref_utts} of {N_UTTS} cfg4 utterances ({frames} frames) in {wall:.1f}s wall, "
                             f"{c.impl} over {cores} processes", "time_basis": "wall time of the pooled map"}
        line = {
            "metric": "mel frames/s (STFT->80-mel log, cache build)", "value": value, "unit": "frames/s",
            "n_gpus": world, "steps": args.steps, "warmup": W, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"cfg4: the fixed corpus of {args.utts} synthetic utterances 1-10 s @22.05 kHz "
                                   f"({int(full_starts[-1]) * 4 / 1e9:.2f} GB samples, {F_total} frames), sharded by utterance over "
                                   f"{world} GPU(s); step = every rank's fused kernel"
                                   + (f" + gather of the shards into rank 0 over NVLink (chunked, overlapped; transport: {gather['headline_transport']})" if world > 1 else "")
                                   + "; inputs >> L2 (126 MB), no flush needed",
                       "n_fft": 1024, "hop": 256, "n_mels": 80, "utterances": args.utts, "frames": F_total,
                       "frames_this_rank": F, "parallelism": f"utterance-sharded x{world}; one exchange: gather of shards"},
            "kernel_only": kernel_only,
            "roofline": {"bound": "hbm", "kernel": "k_stft_mel<0>", "achieved": achieved, "peak": hbm_peak,
                         "unit": "GB/s", "frac": achieved / hbm_peak, "peak_source": peak_src,
                         "alg_bytes_per_frame": ALG_BYTES_PER_FRAME, "kernel_ms": kern_ms,
                         "kernel_ms_max_over_ranks": kern_ms_max, "traffic": NCU_DRAM_BYTES_PER_FRAME * F,
                         "traffic_source": NCU_TRAFFIC_SOURCE,
                         "issue_slots": NCU_ISSUE_NOTE,
                         "note": "fp32-pipe/shared-memory bound by design (SURVEY 0.7): ~25 kFLOP FFT per 1,344 B"},
            "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": args.steps * launches_per_step, "clocks": clocks,
            "parity": parity, "gather": gather, "cfg5": cfg5, "mel_gemm_tc": tc, "frame_features": feat,
            "pyin": pyin_res, "collate": coll, "griffinlim": gl, "length_regulator": lr_res,
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


DUMP_UTTS = 64


def dump_cache_sample(out_dir, cache, plan):
    """Writes ``out_dir/logmel.npy``: the log-mel rows (float32 [rows, 80], corpus order) of DUMP_UTTS utterances drawn
    with a fixed seed from the cache the timed steps built.  The whole cache (~2 GB for cfg4) is too large to keep; the
    sample (<= 18 MB) lets two builds of the project be compared output for output on identical inputs."""
    import torch
    from spev_tts_b200.cache import GatheredCache
    n = len(plan.frames)
    utts = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_UTTS), replace=False))
    gc = GatheredCache(cache, plan)
    rows = torch.cat([gc.utterance(int(u)) for u in utts]).cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "logmel.npy"), rows.astype(np.float32, copy=False))


def measure_pcie(dev, host_in, host_out):
    """Pinned host <-> device copy bandwidth of THIS rank, measured alone and in both directions at once (the e2e
    pipeline overlaps them): the denominator of e2e.roofline."""
    import torch
    n_in = host_in.numel()                         # the WHOLE pinned buffers of the e2e run: on a multi-socket host
    n_out = host_out.numel()                       # different parts of a large pinned allocation can sit on different nodes
    d_in = torch.empty(n_in, dtype=host_in.dtype, device=dev)
    d_out = torch.empty(n_out, dtype=host_out.dtype, device=dev)
    hi, ho = host_in.view(-1)[:n_in], host_out.view(-1)[:n_out]
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    def run(do_in, do_out):
        torch.cuda.synchronize(dev)
        a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
        a.record()
        s1.wait_event(a); s2.wait_event(a)
        if do_in:
            with torch.cuda.stream(s1):
                d_in.copy_(hi, non_blocking=True)
        if do_out:
            with torch.cuda.stream(s2):
                ho.copy_(d_out, non_blocking=True)
        torch.cuda.current_stream(dev).wait_stream(s1); torch.cuda.current_stream(dev).wait_stream(s2)
        b.record(); torch.cuda.synchronize(dev)
        return a.elapsed_time(b) * 1e-3
    run(True, True)
    t_in = run(True, False)
    t_out = run(False, True)
    t_both = run(True, True)
    bi, bo = n_in * hi.element_size(), n_out * ho.element_size()
    return {"h2d_GBps": bi / t_in / 1e9, "d2h_GBps": bo / t_out / 1e9,
            "duplex_GBps": (bi + bo) / t_both / 1e9, "unit": "GB/s", "how": "cudaMemcpyAsync from/to pinned memory, "
            f"{bi >> 20} MiB in / {bo >> 20} MiB out (the e2e run's own buffers, whole), after one warm-up pass, this rank alone"}


def parity_griffinlim(sp, dev, lr_oracle):
    """Spectral-convergence delta of one cfg3 item (80 x 800, 60 iterations, shared initial phase) against the CPU
    oracle -- the north-star's Griffin-Lim tolerance (<= 1e-3), checked inside the measured run."""
    from tests import synth
    y = synth.speechy(seed=300, n=799 * HOP)
    lm = lr_oracle.reference_logmel(y).T.copy()                    # [80, 800]
    ph = synth.init_phase((513, 800), seed=3)
    S = lr_oracle.mel_to_stft(np.exp(lm), sr=SR, n_fft=1024, fmin=0, fmax=8000, lbfgs=True)
    w_ref = lr_oracle.griffinlim(S, n_iter=60, hop_length=HOP, n_fft=1024, init_phase=ph)
    w = sp.Vocoder(n_iter=60, device=dev).infer(lm, init_phase=ph)
    sc_ref, sc = lr_oracle.spectral_convergence(w_ref, S), lr_oracle.spectral_convergence(w, S)
    return {"griffinlim_sc_gpu": sc, "griffinlim_sc_oracle": sc_ref, "griffinlim_sc_delta": abs(sc - sc_ref),
            "griffinlim_sc_tolerance": 1e-3, "griffinlim_case": "1 x [80,800], 60 iterations, shared init phase, NNLS L-BFGS-B on in the oracle"}


def bench_cfg5(sp, dev, hbm_peak, spcache, world, max_over_ranks, sum_over_ranks):
    """configs[4]: LibriTTS-R-shaped multi-speaker 24 kHz variable-length batches across the GPUs of the box.  Every
    rank takes its own set of buckets (seed 5 + rank; weak: more GPUs = more speakers' data): STFT->log-mel on 4,096
    utterances of 1-20 s (mel basis fmax 12 kHz) in one ragged launch, and Griffin-Lim (60 iterations) on a
    256-utterance subset.  Aggregate = sum over ranks / slowest rank's time."""
    import torch
    import torch.distributed as dist
    rank = dist.get_rank() if world > 1 else 0
    res = {"n_gpus": world, "scaling": "weak (per-GPU buckets fixed)"}
    res["logmel"] = _cfg5_logmel(sp, dev, hbm_peak, spcache, rank, world, max_over_ranks, sum_over_ranks)
    res["griffinlim"] = bench_griffinlim_cfg5(sp, dev, hbm_peak, rank, world, max_over_ranks, sum_over_ranks)
    torch.cuda.empty_cache()
    return res


def _cfg5_logmel(sp, dev, hbm_peak, spcache, rank, world, max_over_ranks, sum_over_ranks):
    import torch
    from tests import synth
    lens = synth.lognormal_lengths(seed=5 + rank, n_utts=4096, sr=24000)
    starts = spcache.aligned_offsets(lens)
    g = torch.Generator(device=dev).manual_seed(5 + rank)
    x = torch.randn(int(starts[-1]), generator=g, device=dev) * 0.05
    ctx = sp.Context.get(dev, sr=24000, n_mels=N_MELS)
    batch = sp.make_batch(ctx, n_samples=lens, sample_off=starts)
    out = torch.empty((batch.n_frames, N_MELS), dtype=torch.float32, device=dev)
    for _ in range(3):
        sp.logmel_flat(x, lens, sr=24000, out=out, batch=batch)
    torch.cuda.synchronize(dev)
    a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(5):
        sp.logmel_flat(x, lens, sr=24000, out=out, batch=batch)
    b.record(); torch.cuda.synchronize(dev)
    ms_local = a.elapsed_time(b) / 5
    ms = max_over_ranks(ms_local)
    F = batch.n_frames
    F_all = sum_over_ranks(float(F))
    return {"config": {"workload": f"cfg5: 4096 utterances 1-20 s @24 kHz per GPU ({x.numel() * 4 / 1e9:.2f} GB, {F} frames on rank 0)"},
            "value": F_all / (ms * 1e-3), "unit": "frames/s", "ms_per_step": ms,
            "roofline": {"bound": "hbm", "achieved": ALG_BYTES_PER_FRAME * F / (ms_local * 1e-3) / 1e9, "peak": hbm_peak,
                         "unit": "GB/s", "frac": ALG_BYTES_PER_FRAME * F / (ms_local * 1e-3) / 1e9 / hbm_peak,
                         "note": "rank 0's kernel"}}


def bench_mel_gemm_tc(sp, dev, samples, lens, starts, hbm_peak, fused_out):
    """A/B: the two-kernel tensor-core path (K1' power spectrum -> TMA/tcgen05 3xTF32 mel GEMM) on the
    same cfg4 shard as the fused kernel.  Tensor 'peak' = measured cuBLAS bf16 / 2 (tf32 rate)."""
    import torch
    from spev_tts_b200 import _lib
    ctx = sp.Context.get(dev, sr=SR, n_mels=N_MELS)
    batch = sp.make_batch(ctx, n_samples=lens, sample_off=starts)
    F = batch.n_frames
    power = torch.empty((F, _lib.SPEC_LD), dtype=torch.float32, device=dev)
    out = torch.empty((F, N_MELS), dtype=torch.float32, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream

    def k1():
        _lib.check(ctx.lib.spev_stft_power(ctx.handle, batch.desc, samples.data_ptr(), power.data_ptr(), st))

    def k2():
        _lib.check(ctx.lib.spev_mel_project(ctx.handle, power.data_ptr(), F, out.data_ptr(), 1, 1e-5, -10.0, 2.0, st))

    def t(fn, n=5):
        for _ in range(3):
            fn()
        a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record(); torch.cuda.synchronize(dev)
        return a.elapsed_time(b) / n
    ms1, ms2 = t(k1), t(k2)
    err = float((out - fused_out).abs().max())
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    tf32_peak = (json.load(open(p))["bf16_tflops"] / 2) if os.path.exists(p) else 795.0
    flops = 2.0 * F * 513 * 80 * 3
    bytes_gemm = F * (513 * 4 + 80 * 4)
    return {"config": {"workload": "cfg4 shard, two-kernel tensor-core path (A/B against the fused kernel)"},
            "stft_power_ms": ms1, "mel_project_ms": ms2, "frames_per_s_two_kernel": F / ((ms1 + ms2) * 1e-3),
            "max_abs_diff_vs_fused_logmel": err,
            "roofline": {"bound": "hbm", "kernel": "k_gemm_tf32x3<80,MEL>", "achieved": bytes_gemm / (ms2 * 1e-3) / 1e9,
                         "peak": hbm_peak, "unit": "GB/s", "frac": bytes_gemm / (ms2 * 1e-3) / 1e9 / hbm_peak,
                         "alg_bytes_per_frame": 513 * 4 + 320},
            "tensor": {"achieved_tflops_3xtf32": flops / (ms2 * 1e-3) / 1e12, "peak_tflops_tf32": tf32_peak,
                       "frac": flops / (ms2 * 1e-3) / 1e12 / tf32_peak,
                       "note": "arithmetic intensity 103 FLOP/B (3 passes) < ridge ~125: the projection is HBM-bound"}}


def bench_frame_features(sp, dev, samples, lens, starts, hbm_peak):
    """SURVEY 8(f) row 1 on the cfg4 shard: RMS + spectral centroid (2048-point STFT), one launch."""
    import torch
    ctx = sp.Context.get(dev, sr=SR, n_mels=N_MELS)
    batch = sp.make_batch(ctx, n_samples=lens, sample_off=starts)
    for _ in range(2):
        sp.frame_features_flat(samples, lens, batch=batch)
    a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(3):
        sp.frame_features_flat(samples, lens, batch=batch)
    b.record(); torch.cuda.synchronize(dev)
    ms = a.elapsed_time(b) / 3
    F = batch.n_frames
    return {"config": {"workload": "cfg4 shard: rms + spectral centroid per frame (n_fft=2048, hop=256)"},
            "value": F / (ms * 1e-3), "unit": "frames/s", "ms_per_step": ms,
            "roofline": {"bound": "hbm", "kernel": "k_frame_features", "achieved": 1032.0 * F / (ms * 1e-3) / 1e9,
                         "peak": hbm_peak, "unit": "GB/s", "frac": 1032.0 * F / (ms * 1e-3) / 1e9 / hbm_peak,
                         "alg_bytes_per_frame": 1032,
                         "note": "one full 1024-complex warp FFT per frame (2x the STFT kernel's FFT work): issue-bound"}}


def bench_pyin(sp, dev, hbm_peak, args, with_cpu):
    """SURVEY 8(f) row 2: librosa.pyin (:369) on a cfg4-shaped shard of speech-like signals (the decoder's
    work depends on the voicing pattern, so white noise would flatter it) + whole cache records."""
    import torch
    from spev_tts_b200 import pitch as gp
    from tests import synth
    n_utts = min(2048, args.utts)
    lens = synth.utterance_lengths(seed=4, n_utts=N_UTTS)[:n_utts]
    base = [synth.voiced_unvoiced(seed=i, n=int(lens.max()))[0] for i in range(16)]
    waves = [base[i % 16][: lens[i]] for i in range(n_utts)]
    starts = sp.cache.aligned_offsets(lens)
    host = np.zeros(int(starts[-1]) + 4, dtype=np.float32)
    for w, st in zip(waves, starts[:-1]):
        host[st: st + len(w)] = w
    x = torch.from_numpy(host).to(dev)
    ctx = sp.Context.get(dev, sr=SR, n_mels=N_MELS)
    batch = sp.make_batch(ctx, n_samples=lens, sample_off=starts[:-1])
    pctx = gp.PyinContext.get(dev, sr=SR)
    F = batch.n_frames

    def timed(fn, reps=3):
        keep = [fn(), fn()]                          # the results are GB-sized: warm the allocator for two live copies
        r = fn(); torch.cuda.synchronize(dev)
        del keep
        a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            r = fn()
        b.record(); torch.cuda.synchronize(dev)
        return a.elapsed_time(b) / reps, r
    ms1, yin = timed(lambda: gp.cmnd_flat(x, batch, pctx))
    ms2, (logobs, lunv, vp) = timed(lambda: gp.observe(yin, pctx))
    del yin
    ms3, (states, f0, flag) = timed(lambda: gp.decode(logobs, lunv, batch.frame_off, pctx))
    del logobs, lunv
    ms = ms1 + ms2 + ms3
    audio_s = float(lens.sum()) / SR
    res = {"config": {"workload": f"{n_utts} cfg4-length speech-like utterances ({F} frames, {audio_s:.0f} s of audio): "
                                  "librosa.pyin(fmin=60, fmax=500, hop_length=256) = CMND + observation + Viterbi"},
           "value": F / (ms * 1e-3), "unit": "frames/s", "audio_s_per_s": audio_s / (ms * 1e-3), "ms_per_step": ms,
           "voiced_fraction": float(flag.float().mean()),
           "stages_ms": {"k_yin_cmnd": ms1, "k_pyin_observe": ms2, "k_pyin_viterbi(+finish)": ms3},
           "roofline": {"bound": "hbm", "kernel": "k_pyin_viterbi", "achieved": 2952.0 * F / (ms3 * 1e-3) / 1e9, "peak": hbm_peak,
                        "unit": "GB/s", "frac": 2952.0 * F / (ms3 * 1e-3) / 1e9 / hbm_peak, "alg_bytes_per_frame": 2952,
                        "note": "latency-bound sequential recursion: 736 states x 102 float64 candidates per frame, "
                                "<= 296 utterances in flight; k_yin_cmnd runs at "
                                f"{2 * 1024 * 384 * F / (ms1 * 1e-3) / 1e12:.1f} TFLOP/s fp32 (direct autocorrelation)"}}
    # whole cache records (log-mel + rms/centroid + pYIN + per-phoneme pooling + host duration logic) on a subset
    n_rec = n_utts
    phones = [["<SIL>"] + list("abcdefghijklmnopqrstuvwxyz"[: 5 + i % 20]) + ["<SIL>"] for i in range(n_rec)]
    durs = [sp.uniform_durations(int(lens[i]), len(phones[i])) for i in range(n_rec)]
    stats = {"p_mean": 5.2, "p_std": 0.35, "e_mean": -4.0, "e_std": 2.0, "c_mean": 7.5, "c_std": 0.8}
    sp.build_records(waves[:n_rec], phones[:n_rec], durs[:n_rec], stats, device=dev)      # warm-up at full size: pinned
    torch.cuda.synchronize(dev)                                                           # staging comes from the host allocator's cache afterwards
    t0 = time.perf_counter()
    recs, _ = sp.build_records(waves[:n_rec], phones[:n_rec], durs[:n_rec], stats, device=dev)
    torch.cuda.synchronize(dev)
    wall = time.perf_counter() - t0
    res["cache_records"] = {"utterances": len(recs), "wall_s": wall, "utterances_per_s": len(recs) / wall,
                            "audio_s_per_s": float(lens[:n_rec].sum()) / SR / wall,
                            "note": "host wave list in -> per-utterance record dicts out (incl. H2D, D2H, Python record assembly)"}
    if with_cpu:
        cores = os.cpu_count() or 1
        n_cpu = min(2 * cores, 32)
        fps, aps, cwall = cpu_pyin_throughput(n_cpu, cores)
        res["cpu_baseline"] = {"value": fps, "unit": "frames/s", "audio_s_per_s": aps, "cores": cores, "kind": "port",
                               "sample": f"{n_cpu} cfg4-length utterances in {cwall:.1f}s, oracle/pyin_restated.py over "
                                         f"{min(cores, n_cpu)} processes"}
    return res


def bench_collate(sp, dev, mel, batch, hbm_peak):
    """SURVEY 8(f) row 3: serve training batches from the GPU-resident cfg4 cache (the reference does
    torch.load per item + pad_sequence on the CPU + one H2D copy per batch, spev_real_metrics.py:433-462)."""
    import torch
    rng = np.random.default_rng(9)
    U = batch.n_items
    frames = batch.frames
    phones = np.maximum(2, frames // 9)                       # ~9 frames per phone
    po = np.concatenate([[0], np.cumsum(phones)])
    P = int(po[-1])
    g = torch.Generator(device=dev).manual_seed(9)
    ids = torch.randint(0, 60, (P,), generator=g, device=dev)
    durs = torch.randint(1, 18, (P,), generator=g, device=dev)
    curves = {k: torch.randn(P, generator=g, device=dev) for k in ("pitch", "energy", "breath", "rough", "bright")}
    cache = sp.ResidentCache.from_flat(mel, batch.frame_off, ids, durs, po, curves)
    res = {}
    for B in (16, 256):
        idx = rng.choice(U, B, replace=False)
        for _ in range(3):
            b = cache.collate(idx)
        torch.cuda.synchronize(dev)
        t = time.perf_counter()
        n = 20
        for _ in range(n):
            b = cache.collate(idx)
        torch.cuda.synchronize(dev)
        wall_ms = (time.perf_counter() - t) * 1e3 / n
        nbytes = sum(v.numel() * v.element_size() for v in b.values())
        res[f"B{B}"] = {"wall_ms_per_batch": wall_ms, "output_bytes": nbytes, "GBps_wall": nbytes / (wall_ms * 1e-3) / 1e9,
                        "mel_shape": list(b["mel"].shape)}
    return {"config": {"workload": "cfg4 cache resident on the GPU; collate == reference collate_fn output, one launch"}, **res}


def bench_griffinlim(sp, dev, hbm_peak, args):
    """cfg3: 16 x [80,800] log-mels, 60 iterations.  audio-seconds per second."""
    import torch
    from spev_tts_b200 import _lib
    from tests import synth
    B, T, n_iter = 16, 800, 60
    # configs[2] / SURVEY 8d cfg3: the log-mels of 16 "speechy" signals of 204,544 samples (realistic magnitudes: with
    # white-noise "mels" librosa's NNLS would iterate on every block, which the reference's inputs never do)
    ys = np.stack([synth.speechy(seed=300 + b, n=(T - 1) * HOP) for b in range(B)])
    lm = sp.logmel(torch.from_numpy(ys).to(dev)).transpose(1, 2).contiguous()         # [B, 80, T]
    ctx = sp.Context.get(dev, sr=SR, n_mels=N_MELS, fmin=0.0, fmax=8000.0)
    fb = sp.make_batch(ctx, n_frames=[T] * B, with_chunks=True)
    S = torch.empty((fb.n_frames, _lib.SPEC_LD), dtype=torch.float32, device=dev)
    y = torch.empty(fb.n_out_samples, dtype=torch.float32, device=dev)
    ws = torch.empty(ctx.lib.spev_griffinlim_workspace_bytes(fb.n_frames), dtype=torch.uint8, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def step():
        sp.mel_to_mag_flat(lm.view(-1), fb, ctx, layout=1, is_log=True, out=S)
        sp.griffinlim_flat(S, fb, ctx, n_iter=n_iter, seed=7, out=y, workspace=ws)

    for _ in range(3):
        step()
    torch.cuda.synchronize(dev)
    times = []
    for _ in range(max(3, min(args.steps, 10))):
        flush.zero_()                      # > L2: evict state between timed steps
        a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
        a.record(); step(); b.record()
        torch.cuda.synchronize(dev)
        times.append(a.elapsed_time(b))
    ms = float(np.mean(times))
    audio_s = B * (T - 1) * HOP / SR
    alg = GL_BYTES_PER_FRAME_ITER * fb.n_frames * n_iter + (2372 + 5128) * fb.n_frames
    # e2e: host log-mels in, host waveform out through Vocoder.infer
    voc = sp.Vocoder(n_iter=n_iter, device=dev)
    lm_host = lm.cpu().pin_memory()
    for _ in range(3):
        w = voc.infer(lm_host)
    torch.cuda.synchronize(dev)
    calls = []
    for _ in range(10):
        t = time.perf_counter()
        w = voc.infer(lm_host)                     # returns a host array: the call is synchronous
        calls.append((time.perf_counter() - t) * 1e3)
    e2e_ms = float(np.median(calls))
    # how many of librosa's NNLS blocks iterate on this input (0 for reference-range mels of this length)
    from spev_tts_b200 import spectral as _sp
    fbq = ctx.uniform_batch(B, T)
    tmq = _sp.items_to_rows(lm).view(-1)
    Sq = sp.mel_to_mag_flat(tmq, fbq, ctx, layout=0, is_log=True)
    nnls_blocks = _sp.nnls_refine(Sq, tmq.view(B * T, N_MELS), ctx, B, T, is_log=True)
    return {"metric": "Griffin-Lim audio-s/s", "value": audio_s / (ms * 1e-3), "unit": "audio-s/s",
            "config": {"workload": "cfg3: 16 x [80,800] log-mel, 60 iterations, momentum 0.99; L2 flushed between steps"},
            "ms_per_step": ms, "launches_per_step": 2 * n_iter + 3,
            "roofline": {"bound": "hbm", "kernels": "k_gl_fused (STFT + phase update + inverse transform) + k_ola_pairs",
                         "achieved": alg / (ms * 1e-3) / 1e9,
                         "peak": hbm_peak, "unit": "GB/s", "frac": alg / (ms * 1e-3) / 1e9 / hbm_peak,
                         "alg_bytes_per_frame_iter": GL_BYTES_PER_FRAME_ITER,
                         "note": "algorithmic bytes are SURVEY 8d's two-kernel figure (20,516 B per frame and iteration); the fused "
                                 "iteration keeps the new spectra in registers and moves 17,428 B (y 1,024 + tprev 4,104 + S 2,052 "
                                 "read, tprev 4,104 + pair segment 2,560 written; segment 2,560 read, y 1,024 written)"},
            "e2e": {"value": audio_s / (e2e_ms * 1e-3), "unit": "audio-s/s", "ms_per_step": e2e_ms,
                    "ms_per_call_min_max": [float(min(calls)), float(max(calls))],
                    "api": "Vocoder.infer (host log-mel in, numpy waveform out; mel->linear solved as librosa does: "
                           f"NNLS convergence test on every block, {nnls_blocks} of them iterate)",
                    "h2d_bytes_per_step": int(lm.numel() * 4), "d2h_bytes_per_step": int(w.size * 4)}}


def bench_griffinlim_cfg5(sp, dev, hbm_peak, rank, world, max_over_ranks, sum_over_ranks):
    """cfg5-shaped Griffin-Lim: 256 variable-length utterances per GPU (LibriTTS-R-like log-normal
    lengths 1-20 s at 24 kHz), 60 iterations, one ragged flat batch."""
    import torch
    from spev_tts_b200 import _lib
    from tests import synth
    sr, n_iter = 24000, 60
    lens = synth.lognormal_lengths(seed=5 + rank, n_utts=256, sr=sr)
    frames = 1 + lens // HOP
    ctx = sp.Context.get(dev, sr=sr, n_mels=N_MELS, fmin=0.0, fmax=8000.0)
    fb = sp.make_batch(ctx, n_frames=frames, with_chunks=True)
    g = torch.Generator(device=dev).manual_seed(5 + rank)
    lm = (-4 + 2 * torch.randn(fb.n_frames, N_MELS, generator=g, device=dev)).clamp(-10, 2)   # frame-major
    S = torch.empty((fb.n_frames, _lib.SPEC_LD), dtype=torch.float32, device=dev)
    y = torch.empty(fb.n_out_samples, dtype=torch.float32, device=dev)
    ws = torch.empty(ctx.lib.spev_griffinlim_workspace_bytes(fb.n_frames), dtype=torch.uint8, device=dev)

    def step():
        sp.mel_to_mag_flat(lm.view(-1), fb, ctx, layout=0, is_log=True, out=S)     # tcgen05 GEMM path
        sp.griffinlim_flat(S, fb, ctx, n_iter=n_iter, seed=11, out=y, workspace=ws)

    for _ in range(2):
        step()
    torch.cuda.synchronize(dev)
    a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(3):
        step()
    b.record(); torch.cuda.synchronize(dev)
    ms_local = a.elapsed_time(b) / 3
    ms = max_over_ranks(ms_local)
    audio_all = sum_over_ranks(float(fb.n_out_samples) / sr)
    alg = GL_BYTES_PER_FRAME_ITER * fb.n_frames * n_iter + (2372 + 5128) * fb.n_frames
    return {"config": {"workload": f"cfg5 subset: 256 utterances 1-20 s @24 kHz per GPU ({fb.n_frames} frames on rank 0, state "
                                   f"{fb.n_frames * 10400 / 1e6:.0f} MB >> L2), 60 iterations, ragged flat batch"},
            "value": audio_all / (ms * 1e-3), "unit": "audio-s/s", "ms_per_step": ms,
            "roofline": {"bound": "hbm", "achieved": alg / (ms_local * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                         "frac": alg / (ms_local * 1e-3) / 1e9 / hbm_peak, "note": "rank 0's kernels"}}


def bench_length_regulator(sp, dev, args):
    import torch
    from tests import synth
    x, dur, _ = synth.cfg2_batch(seed=2)
    feats = synth.cfg2_features(seed=2)
    xd, dd = torch.from_numpy(x).to(dev), torch.from_numpy(dur).to(dev)
    fd = [torch.from_numpy(f).to(dev) for f in feats]
    lrm = sp.LengthRegulator()
    for _ in range(3):
        o, ml = lrm(xd, dd)
    p = sp.plan(dd)
    torch.cuda.synchronize(dev)
    t = time.perf_counter()
    n = 20
    for _ in range(n):
        o, ml, cv = sp.regulate_variances(xd, dd, fd)
    torch.cuda.synchronize(dev)
    wall_ms = (time.perf_counter() - t) * 1e3 / n
    a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
    ft = torch.stack(fd)
    a.record()
    for _ in range(n):
        sp.expand(xd, p, ft, sp.VARIANCE_CLAMPS)
    b.record()
    torch.cuda.synchronize(dev)
    k_ms = a.elapsed_time(b) / n
    out_bytes = o.shape[0] * o.shape[1] * (256 + 5) * 4
    # fused variance adaptor (expand + clamp + 5 Conv1d(1,256,3) embeddings + sum, :226-252) vs expand + torch convs
    embs = [torch.nn.Conv1d(1, 256, 3, padding=1).to(dev) for _ in range(5)]
    for _ in range(3):
        sp.variance_adaptor(xd, dd, fd, embs)
    a3 = torch.cuda.Event(enable_timing=True); b3 = torch.cuda.Event(enable_timing=True)
    a3.record()
    for _ in range(n):
        sp.variance_adaptor(xd, dd, fd, embs)
    b3.record()
    torch.cuda.synchronize(dev)
    fused_ms = a3.elapsed_time(b3) / n

    def unfused():
        xe, ml_, ce = sp.regulate_variances(xd, dd, fd)
        di = xe.transpose(1, 2)
        for e_, c_ in zip(embs, ce):
            di = di + e_(c_)
        return di.transpose(1, 2)
    with torch.no_grad():
        for _ in range(3):
            unfused()
        a4 = torch.cuda.Event(enable_timing=True); b4 = torch.cuda.Event(enable_timing=True)
        a4.record()
        for _ in range(n):
            unfused()
        b4.record()
        torch.cuda.synchronize(dev)
    unfused_ms = a4.elapsed_time(b4) / n
    # larger batch (SURVEY 8d: "also measure at B=512"): the expand kernel leaves the latency regime
    rng = np.random.default_rng(12)
    xb = torch.from_numpy(rng.standard_normal((512, 200, 256)).astype(np.float32)).to(dev)
    db = torch.from_numpy(rng.integers(0, 21, (512, 200))).to(dev)
    fb5 = torch.randn(5, 512, 200, device=dev)
    pb = sp.plan(db)
    for _ in range(3):
        ob, _ = sp.expand(xb, pb, fb5, sp.VARIANCE_CLAMPS)
    a2 = torch.cuda.Event(enable_timing=True); b2 = torch.cuda.Event(enable_timing=True)
    a2.record()
    for _ in range(10):
        sp.expand(xb, pb, fb5, sp.VARIANCE_CLAMPS)
    b2.record()
    torch.cuda.synchronize(dev)
    kb_ms = a2.elapsed_time(b2) / 10
    big_bytes = ob.shape[0] * ob.shape[1] * (256 + 5) * 4
    big = {"B": 512, "frames": int(ob.shape[1]), "expand_kernel_ms": kb_ms, "expand_GBps": big_bytes / (kb_ms * 1e-3) / 1e9,
           "output_GB": big_bytes / 1e9}
    # the same forward when the caller knows max_len (training: b['mel'].size(1)): no host sync at all
    maxF = int(o.shape[1])
    for _ in range(3):
        sp.regulate_variances(xd, dd, fd, max_len=maxF)
    torch.cuda.synchronize(dev)
    t = time.perf_counter()
    for _ in range(n):
        sp.regulate_variances(xd, dd, fd, max_len=maxF)
    torch.cuda.synchronize(dev)
    nosync_ms = (time.perf_counter() - t) * 1e3 / n
    # training step: forward + backward of the six LengthRegulator calls (segment-sum kernels)
    xg = xd.clone().requires_grad_(True)
    fg = [f.clone().requires_grad_(True) for f in fd]

    def fwd_bwd():
        oe, _, ce = sp.regulate_variances(xg, dd, fg, max_len=maxF)
        (oe.sum() + sum(c.sum() for c in ce)).backward()
        xg.grad = None
        for f in fg:
            f.grad = None
    for _ in range(3):
        fwd_bwd()
    torch.cuda.synchronize(dev)
    t = time.perf_counter()
    for _ in range(n):
        fwd_bwd()
    torch.cuda.synchronize(dev)
    train_ms = (time.perf_counter() - t) * 1e3 / n
    go = torch.ones_like(o)
    gf = torch.ones((5, o.shape[0], maxF), device=dev)
    ab = torch.cuda.Event(enable_timing=True); bb = torch.cuda.Event(enable_timing=True)
    gx = torch.empty_like(xd); gfe = torch.empty((5,) + tuple(dd.shape), device=dev)
    from spev_tts_b200 import _lib
    from spev_tts_b200.length_regulator import _clamp_arrays
    lo, hi = _clamp_arrays(sp.VARIANCE_CLAMPS, 5)
    st = torch.cuda.current_stream(dev).cuda_stream
    ab.record()
    for _ in range(n):
        _lib.check(_lib.load().spev_lr_expand_backward(go.data_ptr(), 0, 256, gf.data_ptr(), 5, ft.data_ptr(), lo, hi,
                                                       p.cumsum.data_ptr(), p.B, p.T, maxF, gx.data_ptr(), gfe.data_ptr(), st))
    bb.record()
    torch.cuda.synchronize(dev)
    bwd_ms = ab.elapsed_time(bb) / n
    # bucketize + embedding lookup (configs[1] second half): v [32,200] -> [32,200,256], and frame-level [32,maxF]
    v, bins, table = synth.bucketize_case(seed=2)
    vt, bt, tt = (torch.from_numpy(a_).to(dev) for a_ in (v, bins, table))
    vfr = torch.randn(32, maxF, device=dev)

    def t_buck(vv):
        for _ in range(3):
            sp.bucketize_embed(vv, bt, tt)
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            sp.bucketize_embed(vv, bt, tt)
        e1.record()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / n
    bk_ms, bk_fr_ms = t_buck(vt), t_buck(vfr)
    buck = {"phone_level": {"elements": int(vt.numel()), "kernel_ms": bk_ms,
                            "GBps": vt.numel() * 1028 / (bk_ms * 1e-3) / 1e9},
            "frame_level": {"elements": int(vfr.numel()), "kernel_ms": bk_fr_ms,
                            "GBps": vfr.numel() * 1028 / (bk_fr_ms * 1e-3) / 1e9},
            "alg_bytes_per_element": 1028, "note": "4 B read + 1,024 B written per element; table (256 KB) stays in L2"}
    cpu = None
    if not args.no_cpu:
        # same-run CPU legs on this box's host cores: the literal-loop restatement of the reference class
        # (oracle/torch_reference.py, pinned against the class itself) and torch's own bucketize + embedding
        from oracle import torch_reference as tr
        xc, dc = torch.from_numpy(x), torch.from_numpy(dur)
        lr_cpu = tr.LengthRegulator()
        t = time.perf_counter()
        lr_cpu(xc, dc)
        t_h = time.perf_counter() - t
        t = time.perf_counter()
        lr_cpu(torch.from_numpy(feats[0]).unsqueeze(-1), dc)
        t_1 = time.perf_counter() - t
        vc, bc, tc_ = torch.from_numpy(v), torch.from_numpy(bins), torch.from_numpy(table)
        torch.nn.functional.embedding(torch.bucketize(vc, bc), tc_)
        t = time.perf_counter()
        for _ in range(10):
            torch.nn.functional.embedding(torch.bucketize(vc, bc), tc_)
        t_b = (time.perf_counter() - t) / 10
        cpu = {"length_regulator_forward_s": t_h + 5 * t_1, "cores": 1, "kind": "port",
               "sample": f"one H=256 call ({t_h:.2f} s) + 5 x one H=1 call ({t_1:.2f} s each measured once), "
                         "oracle/torch_reference.LengthRegulator (the reference's per-(b,t) .item() loop) on CPU tensors",
               "bucketize_embed_ms": t_b * 1e3, "bucketize_threads": torch.get_num_threads()}
    return {"B512": big, "variance_adaptor_fused_ms": fused_ms, "variance_adaptor_expand_plus_cudnn_ms": unfused_ms,
            "config": {"workload": "cfg2: B=32, T<=200, H=256 + 5 curves (the 6 LengthRegulator calls of one forward)"},
            "forward_ms_wall_incl_one_sync": wall_ms, "forward_ms_wall_max_len_known_no_sync": nosync_ms,
            "expand_kernel_ms": k_ms, "expand_GBps": out_bytes / (k_ms * 1e-3) / 1e9, "frames": int(o.shape[1]),
            "train_fwd_bwd_ms_wall_no_sync": train_ms, "backward_kernels_ms": bwd_ms, "backward_GBps": out_bytes / (bwd_ms * 1e-3) / 1e9,
            "bucketize_embed": buck, "cpu_baseline": cpu}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--utts", type=int, default=N_UTTS, help="utterances per GPU (cfg4: 13100)")
    ap.add_argument("--ref-utts", type=int, default=2048, help="bounded CPU sample (utterances per step)")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--chunks", type=int, default=8, help="chunks per shard for the compute/gather overlap (N > 1)")
    ap.add_argument("--transport", default="best", choices=["best", "nccl", "p2p"],
                    help="gather transport of the headline value at N > 1 (best: the faster of the two, named in the line)")
    ap.add_argument("--reserve-sms", type=int, default=16, help="SMs left to NCCL's kernels while a gather is in flight")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-gl", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a fixed sample of the log-mel cache they built to DIR/logmel.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
