#!/usr/bin/env python
"""bench.py -- tracks/sec analysed (10 s @ 48 kHz) + k-NN queries/sec over 100 k embeddings.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the analysis hot path (PCM16 windows -> log-mel -> student CLAP encoder ->
per-track mean + L2) over one batch of 256 synthetic 10 s tracks per GPU (BASELINE.json configs[1]),
followed, for N > 1, by the single all-gather of the embedding shards (SURVEY 8(e)).

Reported (ONE JSON line on rank 0):
  value     whole-job tracks/s with the batch already resident in HBM (CUDA events, max over ranks)
  e2e       the same metric through the public host API: pinned host PCM16 -> H2D -> kernels -> D2H embeddings,
            all inside the timed region.  value = B200Session.embed_tracks_stream (bulk analysis: two batches in
            flight), sync_call_value = one blocking B200Session.embed_tracks call per step
  roofline  dominant kernel (the tcgen05 pointwise-conv GEMM), tensor bound, from per-launch CUDA
            events recorded by the library inside the timed region; roofline_mel = the fused mel kernel
  knn       k-NN queries/s over 100 000 x 512 (BASELINE.json configs[2]) at batch 4096 / 256 / 1
  cpu_baseline   the oracle (CPU restatement of librosa + onnxruntime, reference libs are not
            installable) timed on this box's host cores on a bounded sample
`--impl reference` times that CPU restatement as the arm itself (rank 0 only).
`--dump-outputs DIR` writes what the last timed step computed to DIR/embeddings.npy (rank 0; inputs and weights are
seeded, so two builds run with the same arguments can be compared output for output).
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
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

TRACKS_PER_GPU = 256
N_SAMPLES = 480000
T_FRAMES = 1001
METRIC = "tracks_per_sec_analysed_10s_48khz"
UNIT = "tracks/s"
WEIGHT_SEED = 0
DUMP_LIMIT_BYTES = 64 << 20


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"hbm_gbs": float(p["hbm_gbs"]), "bf16_tflops": float(p["bf16_tflops"]),
                "bf16_tflops_sustained": float(p.get("bf16_tflops_sustained", p["bf16_tflops"])),
                "source": "MEASURED_PEAKS.json"}
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def _traffic(name):
    """DRAM bytes per launch from the committed ncu --set full capture (profiles/*.json), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            return json.load(f).get(name)
    except Exception:
        return None


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md).  NVML is queried in-process
    (nvidia_ml_py): spawning `nvidia-smi` every 100 ms re-initialises the driver interface for every GPU of the box and
    was seen to stall kernel launches by ~10-20 ms per call (a 12 ms step measured as 13.8 ms); nvidia-smi remains the
    fallback when the module is missing."""

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.rows = []          # (sm_mhz, sm_max_mhz, reasons bitmask or None, [reason names])
        self._stop = threading.Event()
        self._t = None
        self._nvml = None
        self._h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self._max = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._nvml = None

    def _sample_nvml(self):
        n = self._nvml
        sm = float(n.nvmlDeviceGetClockInfo(self._h, n.NVML_CLOCK_SM))
        try:
            mask = int(n.nvmlDeviceGetCurrentClocksEventReasons(self._h))
        except Exception:
            mask = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self._h))
        names = []
        for name, attr in (("hw_slowdown", "nvmlClocksThrottleReasonHwSlowdown"),
                           ("hw_thermal_slowdown", "nvmlClocksThrottleReasonHwThermalSlowdown"),
                           ("sw_thermal_slowdown", "nvmlClocksThrottleReasonSwThermalSlowdown"),
                           ("sw_power_cap", "nvmlClocksThrottleReasonSwPowerCap")):
            bit = getattr(n, attr, None)
            if bit is not None and mask & int(bit):
                names.append(name)
        self.rows.append((sm, self._max, names))

    def _sample_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        out = subprocess.run(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5)
        parts = [x.strip() for x in out.stdout.strip().split(",")]
        if len(parts) >= 6:
            names = [nm for nm, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[2:6])
                     if v.lower().startswith("active")]
            self.rows.append((float(parts[0]), float(parts[1]), names))

    def _run(self):
        while not self._stop.is_set():
            try:
                if self._nvml:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            self._stop.wait(0.02 if self._nvml else 0.25)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=10)
        sm = [r[0] for r in self.rows]
        mx = [r[1] for r in self.rows]
        reasons = sorted({nm for r in self.rows for nm in r[2]})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows), "source": "nvml" if self._nvml else "nvidia-smi"}


# ----------------------------------------------------------------------------------------------
def cpu_reference_tracks_per_sec(n_tracks, state_dict, threads=None):
    """The reference loop restated with the libraries present (SURVEY 8(d) "CPU baseline"): per track
    int16 round trip -> 10 s windows -> per-window numpy mel -> per-window batch-1 encoder (PyTorch CPU
    fp32, all host threads) -> mean + L2.  Returns (tracks/s, seconds, threads)."""
    import torch

    from audiomuse_ai_b200 import corpus
    from oracle import mel as omel, phinet, segments as oseg

    # all physical host cores, like the reference's onnxruntime session default (torchrun pins
    # OMP_NUM_THREADS=1: override; logical-CPU counts oversubscribe and run ~30x slower)
    if not threads:
        try:
            import psutil
            threads = psutil.cpu_count(logical=False) or 0
        except Exception:
            threads = 0
        threads = threads or max(1, (os.cpu_count() or 2) // 2)
    torch.set_num_threads(threads)
    model = phinet.StudentCLAPAudio()
    model.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in state_dict.items()}, strict=False)
    model.eval()
    pcm = corpus.synth_pcm_batch(n_tracks, start=100)
    # untimed warm-up (thread pools, allocator)
    phinet.embed_segments(model, omel.compute_mel_spectrogram(corpus.pcm16_to_float(pcm[0])[:96000]))
    t0 = time.perf_counter()
    for i in range(n_tracks):
        x, _ = oseg.int16_round_trip(corpus.pcm16_to_float(pcm[i]))
        embs = [phinet.embed_segments(model, omel.compute_mel_spectrogram(s)) for s in oseg.segment_audio(x)]
        oseg.pool_segments(np.vstack(embs))
    dt = time.perf_counter() - t0
    return n_tracks / dt, dt, torch.get_num_threads()


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    from audiomuse_ai_b200 import weights
    sd = weights.random_state_dict(WEIGHT_SEED)
    sample = 8  # tracks per step: ~2.5 s of host work, so any --steps the driver picks ends within minutes
    for _ in range(max(args.warmup, 0)):
        cpu_reference_tracks_per_sec(1, sd)
    vals, secs, cores = [], 0.0, os.cpu_count()
    for _ in range(max(args.steps, 1)):
        v, dt, cores = cpu_reference_tracks_per_sec(sample, sd)
        vals.append(v)
        secs += dt
    value = sample * len(vals) / secs
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * secs / len(vals),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[1]: synthetic 10s@48kHz tracks -> mel + CLAP embed, reference loop "
                               "(one window per call) on host cores", "tracks_per_step": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{sample} tracks per step x {len(vals)} steps; numpy mel + PyTorch-CPU "
                                   "fp32 encoder, batch 1 per window (librosa/onnxruntime not installable)",
                         "threads": "torch.set_num_threads(physical cores), pinned for every step",
                         "per_step_values": [round(v, 3) for v in vals],
                         "run_to_run_spread": (max(vals) / min(vals)) if vals and min(vals) > 0 else None},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def dump_embeddings(out_dir, emb):
    """Writes the f32[n, dim] embeddings a caller of the timed path receives as out_dir/embeddings.npy.  Above
    DUMP_LIMIT_BYTES a fixed seeded sample of rows is written instead, with their row numbers in embeddings_rows.npy."""
    os.makedirs(out_dir, exist_ok=True)
    emb = np.ascontiguousarray(emb, dtype=np.float32)
    max_rows = DUMP_LIMIT_BYTES // (emb.shape[1] * 4 + 8)
    if len(emb) > max_rows:
        rows = np.sort(np.random.default_rng(0).choice(len(emb), max_rows, replace=False))
        emb = emb[rows]
        np.save(os.path.join(out_dir, "embeddings_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "embeddings.npy"), emb)


# ----------------------------------------------------------------------------------------------
def run_scale_sections(args, sess, plan, pcm_dev, offs_dev, dev, rank, world, barrier):
    """Three measurements that involve everything AFTER the per-track analysis, at `world` GPUs (device time through
    CUDA events, max over ranks; collectives are NCCL through torch.distributed):

    strong_scaling   a FIXED library of --library-tracks 10 s tracks, sharded contiguously over the ranks (each rank
                     streams its shard through the resident 256-track batch), one all-gather of the embedding shards,
                     index build from the gathered DEVICE buffer on every rank.  tracks/s of the whole job.
    knn_sharded      config 3 at N GPUs: 100 k x 512 library rows generated shard-wise on the ranks, all-gathered,
                     Index.from_device (no host round trip); 10 000 queries dealt round-robin to the ranks, one
                     all-gather of the (id, distance) pairs; ids checked against a single-rank answer.
    kmeans_sharded   config 4 at N GPUs: --kmeans-rows x 512 rows sharded as produced, k = 128, 20 fixed Lloyd
                     iterations (am_kmeans_plan_step per rank + ONE all-reduce of [k, d] sums and [k] counts per
                     iteration): ms per iteration and the all-reduce's share."""
    import torch
    import torch.distributed as dist

    from audiomuse_ai_b200 import corpus, dist as amdist, voyager_compat as vc

    out = {}
    n_batch = int(offs_dev.numel()) - 1
    stream = torch.cuda.current_stream(dev)

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        r = fn()
        e1.record(stream)
        barrier()
        return amdist.max_over_ranks(e0.elapsed_time(e1), dev), r

    # ---------------- strong scaling: fixed library
    try:
        n_lib = int(args.library_tracks)
        lo, hi = amdist.shard_bounds(n_lib, rank, world)
        n_mine = hi - lo
        plen = amdist.padded_shard_len(n_lib, world)
        emb = torch.zeros((plen, sess.embedding_dim), dtype=torch.float32, device=dev)
        scratch = torch.empty((n_batch, sess.embedding_dim), dtype=torch.float32, device=dev)
        full = torch.empty((world * plen, sess.embedding_dim), dtype=torch.float32, device=dev)

        def analyse_and_gather():
            for b0 in range(0, n_mine, n_batch):
                nb = min(n_batch, n_mine - b0)
                dst = emb[b0:b0 + nb] if nb == n_batch else scratch
                sess.embed_tracks_dev(plan, pcm_dev.data_ptr(), N_SAMPLES, offs_dev.data_ptr(), nb, nb, dst.data_ptr(),
                                      stream.cuda_stream)
                if nb != n_batch:
                    emb[b0:b0 + nb].copy_(scratch[:nb])
            if world > 1:
                dist.all_gather_into_tensor(full, emb)
                return full
            return emb

        analyse_and_gather()  # warm-up (workspace sizes, NCCL channel)
        ms_a, lib_dev = timed(analyse_and_gather)
        t0 = time.perf_counter()
        if world > 1 and n_lib % world:   # drop the per-shard padding rows
            lib_dev = torch.cat([lib_dev[r * plen:r * plen + (amdist.shard_bounds(n_lib, r, world)[1] - amdist.shard_bounds(n_lib, r, world)[0])]
                                 for r in range(world)])
        idx = vc.Index.from_device(lib_dev[:n_lib], vc.Space.Cosine)
        torch.cuda.synchronize(dev)
        build_s = amdist.max_over_ranks(time.perf_counter() - t0, dev)
        total_s = ms_a / 1e3 + build_s
        out["strong_scaling"] = {
            "library_tracks": n_lib, "tracks_per_rank": n_mine, "analysis_plus_gather_ms": ms_a,
            "index_build_ms": 1e3 * build_s, "tracks_per_s_whole_job": n_lib / total_s, "scaling": "strong",
            "collective": f"one all_gather_into_tensor of f32[{plen}, {sess.embedding_dim}] per rank" if world > 1 else "none",
            "note": "every rank streams its contiguous shard through the resident 256-track synthetic batch"}
        del idx, full, emb
    except Exception as e:
        out["strong_scaling"] = {"error": str(e)}

    # ---------------- k-NN: gathered device library, sharded queries
    try:
        x = corpus.knn_library(100_000, 512, 1234)          # same rows on every rank (seeded); each uploads ITS shard
        lo, hi = amdist.shard_bounds(len(x), rank, world)
        lib_dev = amdist.all_gather_embeddings(torch.from_numpy(x[lo:hi]).to(dev), len(x))
        idx = vc.Index.from_device(lib_dev, vc.Space.Cosine)
        q = corpus.knn_queries(x, 9_000, 1_000, 4321)
        amdist.sharded_knn_query(idx, q, 50)               # warm-up with the timed shapes (score buffers, NCCL channel)
        dts = []
        for _ in range(3):
            barrier()
            t0 = time.perf_counter()
            ids, dd = amdist.sharded_knn_query(idx, q, 50)
            dts.append(amdist.max_over_ranks(time.perf_counter() - t0, dev))
        dt = sorted(dts)[1]                                # median of three calls
        ok = True
        if rank == 0:
            ref_ids, _ = idx.query(q, 50)
            ok = bool(np.array_equal(ids, np.asarray(ref_ids, dtype=np.int64)))
        out["knn_sharded"] = {"library": "100000 x 512 gathered on device (Index.from_device)", "queries": len(q), "k": 50,
                              "queries_per_s": len(q) / dt, "ms_total": 1e3 * dt, "ms_all_calls": [round(1e3 * t, 3) for t in dts],
                              "ids_equal_single_rank_answer": ok,
                              "collective": "all_gather of the [nq/W, 50] (id, distance) pairs" if world > 1 else "none"}
        del idx, lib_dev
    except Exception as e:
        out["knn_sharded"] = {"error": str(e)}

    # ---------------- k-means: rows sharded, one all-reduce per Lloyd iteration
    try:
        n_rows, d, k, iters = int(args.kmeans_rows), 512, 128, 20
        lo, hi = amdist.shard_bounds(n_rows, rank, world)
        g = torch.Generator(device=dev)
        g.manual_seed(7)
        centers_true = torch.nn.functional.normalize(torch.randn((k, d), generator=g, device=dev), dim=1)
        g.manual_seed(1000 + rank)
        lab = torch.randint(0, k, (hi - lo,), generator=g, device=dev)
        xk = torch.nn.functional.normalize(centers_true[lab] + (0.5 / d ** 0.5) * torch.randn((hi - lo, d), generator=g, device=dev), dim=1)
        del lab
        init = xk[:k].clone()
        if world > 1:
            dist.broadcast(init, 0)
        tm = {}
        amdist.kmeans_lloyd_sharded(xk, init, max_iter=2, tol=None)          # warm-up
        barrier()
        t0 = time.perf_counter()
        _, _, inertia, it = amdist.kmeans_lloyd_sharded(xk, init, max_iter=iters, tol=None, timing=tm)
        wall = amdist.max_over_ranks(time.perf_counter() - t0, dev)
        assign_ms = amdist.max_over_ranks(tm["assign_ms"], dev) / iters
        ar_ms = amdist.max_over_ranks(tm["allreduce_ms"], dev) / iters
        out["kmeans_sharded"] = {
            "rows_total": n_rows, "rows_per_rank": hi - lo, "d": d, "k": k, "iterations": iters,
            "ms_per_iteration_device": assign_ms + ar_ms, "assign_and_partial_sums_ms": assign_ms, "allreduce_ms": ar_ms,
            "allreduce_share": ar_ms / max(assign_ms + ar_ms, 1e-9), "wall_ms_per_iteration_incl_split_and_final_pass": 1e3 * wall / iters,
            "inertia": inertia, "tensor_cores": bool(tm.get("tensor_cores")),
            "collective": f"all_reduce(sum) of f32[{k}, {d}] + f32[{k}] per iteration" if world > 1 else "none",
            "hbm_bound_ms_per_iteration": 2.0 * (hi - lo) * d * 4 / (_peaks()["hbm_gbs"] * 1e9) * 1e3}
        # roofline of the Lloyd iteration: two passes over the rows (split-bf16 copy for the assignment, fp32 rows for the
        # partial sums) = 2 N d 4 bytes against the measured HBM peak
        km = out["kmeans_sharded"]
        km["roofline"] = {"bound": "hbm", "achieved": 2.0 * (hi - lo) * d * 4 / (assign_ms * 1e-3) / 1e9, "peak": _peaks()["hbm_gbs"],
                          "unit": "GB/s", "frac": km["hbm_bound_ms_per_iteration"] / max(assign_ms, 1e-9)}
        del xk
    except Exception as e:
        out["kmeans_sharded"] = {"error": str(e)}
    torch.cuda.empty_cache()
    return out


# ----------------------------------------------------------------------------------------------
def run_b200(args):
    import torch

    import __graft_entry__ as ge
    from audiomuse_ai_b200 import _lib, clap_analyzer as ca, corpus, dist as amdist, voyager_compat as vc, weights

    rank, local_rank, world = amdist.init_process_group()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this framework has no CPU path (use --impl reference)")
    if not os.path.exists(_lib.LIB_PATH):
        ge.build()
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    numa_node = amdist.bind_to_gpu_numa_node(local_rank) if world > 1 else None   # before the pinned buffers exist
    _lib.check(_lib.load().am_init(local_rank))
    peaks = _peaks()

    sd = weights.random_state_dict(WEIGHT_SEED)
    sess = ca.B200Session.from_state_dict(sd)
    plan = ca.MelPlan()
    n_tracks = args.tracks
    min_warm = 1 if args.profile_mode else 3
    pcm_host = torch.from_numpy(corpus.synth_pcm_batch(n_tracks, start=1000 * rank)).pin_memory()
    offs_host = torch.arange(n_tracks + 1, dtype=torch.int32).pin_memory()
    pcm_dev = pcm_host.to(dev, non_blocking=True)
    offs_dev = offs_host.to(dev, non_blocking=True)
    out_dev = torch.empty((n_tracks, sess.embedding_dim), dtype=torch.float32, device=dev)
    gathered = torch.empty((world * n_tracks, sess.embedding_dim), dtype=torch.float32, device=dev) if world > 1 else None
    stream = torch.cuda.current_stream(dev)

    def step_device():
        sess.embed_tracks_dev(plan, pcm_dev.data_ptr(), N_SAMPLES, offs_dev.data_ptr(), n_tracks, n_tracks,
                              out_dev.data_ptr(), stream.cuda_stream)
        if world > 1:
            torch.distributed.all_gather_into_tensor(gathered, out_dev)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(max(args.warmup, min_warm)):
        step_device()
    barrier()

    # ---- timed region: K steps, device-resident inputs (246 MB of PCM16 per step > 126 MB L2)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    _lib.profile_enable(True)
    _lib.profile_report()  # clear
    launches0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        step_device()
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    launches = _lib.launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_embeddings(args.dump_outputs, (gathered if world > 1 else out_dev).cpu().numpy())
    prof = _lib.profile_report()
    _lib.profile_enable(False)
    clocks = sampler.stop() if sampler else None
    ms = amdist.max_over_ranks(ms, dev)
    value = world * n_tracks * args.steps / (ms / 1000.0)

    # ---- end to end through the host API (pinned host PCM -> H2D -> kernels -> D2H)
    pcm_np, offs_np = pcm_host.numpy(), offs_host.numpy()
    e2e_value = e2e_sync = None
    if not args.skip_e2e:
        for _ in range(2):
            sess.embed_tracks(pcm_np, offs_np)
        # (a) one synchronous call per step
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            emb_host = sess.embed_tracks(pcm_np, offs_np)
        torch.cuda.synchronize(dev)
        e2e_sync = world * n_tracks * args.steps / amdist.max_over_ranks(time.perf_counter() - t0, dev)
        # (b) the bulk-analysis call: batches streamed through the session (two in flight: the next batch's
        #     H2D and early blocks run under this batch's tail).  Every step still copies its PCM from pinned
        #     host memory and reads its embeddings back; the timed region ends when the last result is on the host.
        list(sess.embed_tracks_stream([(pcm_np, offs_np)] * 2))
        barrier()
        t0 = time.perf_counter()
        for emb_host in sess.embed_tracks_stream((pcm_np, offs_np) for _ in range(args.steps)):
            pass
        torch.cuda.synchronize(dev)
        e2e_s = amdist.max_over_ranks(time.perf_counter() - t0, dev)
        e2e_value = world * n_tracks * args.steps / e2e_s
        # the device-resident result and the host-API result are the same numbers
        assert np.allclose(emb_host, out_dev.cpu().numpy(), atol=1e-6), "host API and device path disagree"

    # ---- the post-gather half of the path at N GPUs (BASELINE.json configs[2-4], SURVEY 8(e)); every rank takes part
    scale = {}
    if not args.skip_scale:
        scale = run_scale_sections(args, sess, plan, pcm_dev, offs_dev, dev, rank, world, barrier)

    if rank != 0:
        return
    # ---- rooflines from the per-launch events recorded inside the timed region
    gemm_fl, fused_fl, fused_by = sess.flops_split(T_FRAMES)
    def kernel_rec(substr):
        ms = sum(v["ms"] for k, v in prof.items() if substr in k)
        cnt = sum(v["count"] for k, v in prof.items() if substr in k)
        return {"ms": ms, "count": cnt}

    gemm = kernel_rec("gemm_tcgen05_kernel")
    # the inverted-residual blocks that run fused: channel-per-lane kernel (blocks with an expansion conv) and the
    # pixel-per-lane kernel (block 0, no expansion); flops_split() counts both as "fused"
    fusedk = kernel_rec("fused_block")
    fused_parts = {k.split("(")[0].split("::")[-1].split("<")[0]: round(v["ms"] / max(args.steps, 1), 4)
                   for k, v in prof.items() if "fused_block" in k}
    peak_tf = peaks["bf16_tflops_sustained"]

    def tensor_roofline(name, rec, flops_per_window, note):
        tf = flops_per_window * n_tracks * args.steps / (rec["ms"] / 1000.0) / 1e12 if rec["ms"] > 0 else 0.0
        return {"kernel": f"{name} ({note})", "bound": "tensor", "achieved": tf, "peak": peak_tf,
                "unit": "TFLOP/s", "frac": tf / peak_tf, "traffic": _traffic(name), "launches": rec["count"],
                "share_of_step": rec["ms"] / (ms if ms > 0 else 1.0), "flops_per_window": flops_per_window,
                "peak_source": peaks["source"] + " bf16_tflops_sustained (kernel timed inside a long step)"}

    r_gemm = tensor_roofline("gemm_tcgen05_kernel", gemm, gemm_fl, "unfused pointwise convs, bf16 -> fp32 TMEM")
    r_fused = tensor_roofline("fused_block_t_kernel + fused_block_kernel", fusedk, fused_fl,
                              "expand + depthwise + project per block, tcgen05 + CUDA cores")
    r_fused["ms_per_step_by_kernel"] = fused_parts
    if fusedk["ms"] > 0:  # the same kernel against the HBM roofline (block input + output only)
        gbs = fused_by * n_tracks * args.steps / (fusedk["ms"] / 1000.0) / 1e9
        r_fused["hbm_view"] = {"achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
                               "algorithmic_bytes_per_window": fused_by}
    roofline = r_fused if fusedk["ms"] >= gemm["ms"] else r_gemm
    roofline_other = r_gemm if roofline is r_fused else r_fused
    mel = kernel_rec("mel_kernel")
    mel_bytes = (N_SAMPLES * 2 + 128 * T_FRAMES * 4) * n_tracks * args.steps
    mel_gbs = mel_bytes / (mel["ms"] / 1000.0) / 1e9 if mel["ms"] > 0 else 0.0
    roofline_mel = {"kernel": "mel_kernel<int16>", "bound": "hbm", "achieved": mel_gbs, "peak": peaks["hbm_gbs"],
                    "unit": "GB/s", "frac": mel_gbs / peaks["hbm_gbs"], "traffic": _traffic("mel_kernel"),
                    "launches": mel["count"], "share_of_step": mel["ms"] / (ms if ms > 0 else 1.0),
                    "algorithmic_bytes_per_window": N_SAMPLES * 2 + 128 * T_FRAMES * 4}
    # the same kernel against the fp32 FMA peak: 1001 frames x (5 N log2 N / 2 real-FFT flops + power + sparse mel + log),
    # SURVEY 8(d); peak = SMs x 128 FMA lanes x 2 flop x max SM clock (nominal: no measured fp32 figure in MEASURED_PEAKS.json)
    mel_flops = T_FRAMES * (56320 + 3 * 1025 + 2 * 1176 + 128)
    sm_mhz = (clocks or {}).get("sm_max_mhz") or 1965.0
    fp32_peak = torch.cuda.get_device_properties(dev).multi_processor_count * 128 * 2 * sm_mhz * 1e6 / 1e12
    mel_tf = mel_flops * n_tracks * args.steps / (mel["ms"] / 1000.0) / 1e12 if mel["ms"] > 0 else 0.0
    roofline_mel["compute_view"] = {"achieved": mel_tf, "peak": fp32_peak, "unit": "TFLOP/s (fp32)", "frac": mel_tf / fp32_peak,
                                    "flops_per_window": mel_flops, "peak_source": "nominal: SMs x 128 x 2 x max SM clock"}
    kernel_ms = {k: round(v["ms"] / args.steps, 4) for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])}

    # ---- k-NN (BASELINE.json configs[2]): 100k x 512 library
    knn = {}
    try:
        if args.skip_knn:
            raise RuntimeError("skipped (--skip-knn)")
        x = corpus.knn_library(100_000, 512, 1234)
        q = corpus.knn_queries(x, 3840, 256, 4321)
        idx = vc.Index(vc.Space.Cosine, num_dimensions=512, M=64, ef_construction=1024)
        idx.add_items(x)
        idx.query(q[:256], 50)
        idx.query(q[:4096], 50)  # warm the stream-ordered scratch pool
        for nq, reps in ((4096, 3), (256, 5), (1, 50)):
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            for r in range(reps):
                idx.query(q[:nq] if nq > 1 else q[r], 50)
            knn[f"qps_batch{nq}"] = nq * reps / (time.perf_counter() - t0)
        _lib.profile_enable(True)
        _lib.profile_report()
        idx.query(q[:4096], 50)
        knn["kernel_ms_batch4096"] = {k: round(v["ms"], 3) for k, v in _lib.profile_report().items()}
        idx.query(q[0], 50)
        knn["kernel_ms_batch1"] = {k: round(v["ms"], 4) for k, v in _lib.profile_report().items()}
        _lib.profile_enable(False)
        t0 = time.perf_counter()
        for r in range(5):
            s = x @ q[r]
            top = np.argpartition(-s, 50)[:50]
            top[np.argsort(-s[top])]
        knn["cpu_numpy_qps_batch1"] = 5 / (time.perf_counter() - t0)
        knn["library"] = "100000 x 512 f32 unit vectors, k=50, host-API timing incl. H2D/D2H"
        # rooflines of the two regimes (VERDICT r1 item 4): the batch is a tensor-core GEMM (2 nq N d flop) followed by
        # the selection; a single query is one pass over the bf16 copy of the library (N d 2 bytes)
        k4, k1 = knn["kernel_ms_batch4096"], knn["kernel_ms_batch1"]
        g_ms = sum(v for k, v in k4.items() if "gemm" in k)
        s1_ms = sum(v for k, v in k1.items() if "score" in k)
        if g_ms > 0:
            tf = 2.0 * 4096 * 100_000 * 512 / (g_ms * 1e-3) / 1e12
            knn["roofline_batch4096"] = {"kernel": "gemm_tcgen05_kernel (bf16 scores + per-32 maxima)", "bound": "tensor",
                                          "achieved": tf, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                                          "frac": tf / peaks["bf16_tflops_sustained"],
                                          "selection_ms": sum(v for k, v in k4.items() if "select" in k),
                                          "all_kernels_ms": sum(k4.values())}
        if s1_ms > 0:
            gbs = 100_000 * 512 * 2 / (s1_ms * 1e-3) / 1e9
            knn["roofline_batch1"] = {"kernel": "score_bf16_small_kernel (one pass over the bf16 library copy)", "bound": "hbm",
                                      "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
                                      "selection_ms": sum(v for k, v in k1.items() if "select" in k),
                                      "all_kernels_ms": sum(k1.values())}
    except Exception as e:  # the analysis line is still valid
        knn["error"] = str(e)

    # ---- CPU baseline (bounded sample) on this box's host cores
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        v, dt, cores = cpu_reference_tracks_per_sec(args.cpu_sample, sd)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{args.cpu_sample} of the 256 tracks ({dt:.1f} s); numpy mel + PyTorch-CPU fp32 encoder, "
                         "one window per call like tasks/clap_analyzer.py:530-535 (librosa/onnxruntime absent)"}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, min_warm), "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"configs[1]: batch={n_tracks} synthetic 10s@48kHz tracks per GPU -> mel + CLAP embed",
                   "tracks_per_gpu": n_tracks, "numa_node_of_rank0": numa_node, "window_samples": N_SAMPLES, "encoder": "PhiNet student "
                   "alpha=3.0 beta=0.75 t0=6 N=8 (8.3 M params, random init seed 0)",
                   "l2": "inputs larger than L2 (245.8 MB PCM16 per step vs 126 MB)",
                   "parallelism": f"dp{world} (tracks sharded, one all-gather of embeddings per step)"},
        "e2e": {"value": e2e_value, "unit": UNIT, "api": "B200Session.embed_tracks_stream (pipelined, 2 batches in flight)",
                "sync_call_value": e2e_sync, "h2d_bytes_per_step": int(pcm_np.nbytes + offs_np.nbytes),
                "d2h_bytes_per_step": int(n_tracks * sess.embedding_dim * 4)},
        "gpu_launches": int(launches),
        "roofline": roofline, "roofline_2nd": roofline_other, "roofline_mel": roofline_mel,
        "kernel_ms_per_step": kernel_ms,
        "knn": knn, "clocks": clocks, "cpu_baseline": cpu,
    }
    line.update(scale)
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-sample", type=int, default=32)  # ~10 s of host work at ~3 tracks/s
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--tracks", type=int, default=TRACKS_PER_GPU, help="tracks per GPU per step (default 256)")
    ap.add_argument("--skip-knn", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--skip-scale", action="store_true", help="skip the strong-scaling / sharded k-NN / sharded k-means sections")
    ap.add_argument("--library-tracks", type=int, default=100_000, help="fixed library size of the strong-scaling section")
    ap.add_argument("--kmeans-rows", type=int, default=1_000_000)
    ap.add_argument("--profile-mode", action="store_true",
                    help="for runs under ncu: honour --warmup < 3; the printed numbers are NOT bench values")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the embeddings of the last timed step to DIR/embeddings.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)
    try:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.destroy_process_group()
    except Exception:
        pass


if __name__ == "__main__":
    main()
