#!/usr/bin/env python
"""bench.py -- throughput of diart's per-chunk hot path on B200 (see DESIGN.md, "Measurement").

    python bench.py --gpus 1 --steps 10 --warmup 3                      # this repo's CUDA path
    python bench.py --impl reference --gpus 1 --steps 3 --warmup 1      # the CPU path (oracle port)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W       # N independent streams, 1/GPU
    python bench.py --steps 10 --warmup 3 --dump-outputs DIR            # + the last timed step's results as DIR/*.npy

Metric (BASELINE.json): stream audio-seconds per second = chunks/s x 0.5 s, 5 s windows @ 16 kHz,
0.5 s step, batch 256.  A step is one pass of the fused pipeline (segmentation -> OSP -> embedding ->
normalisation -> clustering, reference blocks/diarization.py:177-203) over one batch of 256 windows.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark runs from a tree it must leave as it found it (possibly read-only)

CHUNK, STEP, SR = 80000, 8000, 16000
STEP_SECONDS = STEP / SR
METRIC = "audio-seconds/sec (real-time factor) at 5s/0.5s step, batch 256"
UNIT = "stream audio-seconds per second"
WORKLOAD = ("configs[2]: full SpeakerDiarization hot path incl. OnlineSpeakerClustering, batch=256 windows of "
            "5 s @ 16 kHz (0.5 s step) of one synthetic stream per GPU, max_speakers=20, pyannote/segmentation + "
            "pyannote/embedding architectures with seeded random-init weights")

# algorithmic FLOPs per chunk of every dense kernel (SURVEY.md 8(a)/(d)); a launch processes B chunks
FLOPS_PER_CHUNK = {
    "sinc0": 2 * 251 * 80 * 7975,
    "sinc_conv1": 2 * 400 * 60 * 2654,
    "sinc_conv2": 2 * 300 * 60 * 880,
    "lstm_inproj": 2 * 1024 * 293 * (60 + 3 * 256) / 4,      # mean over the 4 layers (one launch each)
    "lstm_rec": 2 * 128 * 512 * 2 * 293,
    "seg_linear": 2 * 293 * (256 * 128 + 128 * 128) / 2,
    "tdnn1": 2 * 300 * 512 * 289,
    "tdnn2": 2 * 1536 * 512 * 285,
    "tdnn3": 2 * 1536 * 512 * 279,
    "tdnn4": 2 * 512 * 512 * 279,
    "tdnn5": 2 * 512 * 1500 * 279,
    "emb_linear": 2 * 3000 * 512 * 3,
}
# algorithmic HBM bytes per chunk and launch of the streaming kernels (DESIGN.md section 3): operand planes in + rows out
HBM_BYTES_PER_CHUNK = {
    # mean over the 4 layers: A hi/lo planes 293 x (64 + 3 x 256) / 4 x 2 B x 2, float32 gate rows 293 x 1024 x 4 B out
    "lstm_inproj": 293 * (64 + 3 * 256) / 4 * 2 * 2 + 293 * 1024 * 4,
    # (both nets / all call sites pooled) float32 map in, two 16-bit planes out: mean over the 7 launches of a step
    "split16": (2 * (2658 * 80 * 4 + 2658 * 128 * 4) + 2 * (2654 * 64 * 4 + 884 * 64 * 4) + 2 * (880 * 64 * 4 + 293 * 64 * 4)
                + 3 * (3000 + 3008) * 4) / 7,
    # sequential clustering: scores + embeddings in, speaker map out (latency-bound: 256 dependent chunks per launch)
    "cluster_step": 293 * 3 * 4 + 3 * 512 * 4 + 3 * 4,
}
# compulsory HBM bytes per chunk of the whole step: waveform in, seg + emb out (SURVEY.md 8(d))
BYTES_PER_CHUNK = 80000 * 4 + 293 * 3 * 4 + 3 * 512 * 4
STEP_FLOPS_PER_CHUNK = 3.359e9      # SURVEY.md 8(d): segmentation 1.312 + embedding (de-duplicated trunk) 2.047 GFLOP
# variant B (WeSpeaker ResNet34, SURVEY.md 8(a) A8'): algorithmic FLOPs per chunk of all launches under one tag
FLOPS_PER_CHUNK_STEP = {
    "fbank_dft": 2 * 498 * 400 * 514,
    "resnet_l1": 6 * 2 * 39840 * 32 * 32 * 9,
    "resnet_l2": 2 * 9960 * 64 * (32 * 9 + 32 + 7 * 64 * 9),
    "resnet_l3": 2 * 2500 * 128 * (64 * 9 + 64 + 11 * 128 * 9),
    "resnet_l4": 2 * 630 * 256 * (128 * 9 + 128 + 5 * 256 * 9),
}
STEP_FLOPS_PER_CHUNK_WESPEAKER = 1.312e9 + sum(FLOPS_PER_CHUNK_STEP.values()) + 3 * (2 * 5120 * 256 + 2 * 2 * 2560 * 63)


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "tf": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "src": "measured"}
    return {"hbm_gbs": 6650.0, "tf": 1400.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None
        self.stamps, self.t_mark = [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "20"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])
            self.stamps.append(time.monotonic())

    def mark(self):
        """samples from here on count (the sampler is started before the warm-up: on an 8-GPU box nvidia-smi needs longer than
        a 70 ms timed region to deliver its first line)"""
        self.t_mark = time.monotonic()

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            self.thread.join(timeout=2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        window = "timed region"
        if self.t_mark is not None:
            inside = [r for r, t in zip(self.rows, self.stamps) if t >= self.t_mark]
            if inside:
                self.rows = inside
            else:
                window = "warm-up + timed region (same load; no sample fell inside the timed region)"
        sm = [float(r[1]) for r in self.rows if len(r) >= 9]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 9:
                continue
            for name, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(self.rows[0][2]), "reasons": sorted(reasons),
                "samples": len(sm), "window": window}


def make_stream_batches(rank: int, n_batches: int, batch: int) -> np.ndarray:
    from diart_b200 import synth

    n_chunks = n_batches * batch
    stream = synth.synth_audio(CHUNK + STEP * (n_chunks - 1), seed=1234 + rank)
    return np.stack([synth.windows(stream, batch, first=j * batch) for j in range(n_batches)])


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(directory: str, arrays: dict):
    """Writes what the timed path returned in its last step, {name: array with windows on axis 0}, as directory/<name>.npy in
    float32 (float64 arrays stay float64).  When that exceeds DUMP_LIMIT_BYTES in all, every array keeps the same seeded sample
    of windows, whose indices are written as window_index.npy."""
    arrays = {k: np.asarray(v, dtype=np.float64 if np.asarray(v).dtype == np.float64 else np.float32) for k, v in arrays.items()}
    n = len(next(iter(arrays.values())))
    per_window = sum(a.nbytes for a in arrays.values()) // n + 8
    if n * per_window > DUMP_LIMIT_BYTES - 4096:          # (4096: room for the .npy headers)
        keep = np.sort(np.random.default_rng(0).choice(n, (DUMP_LIMIT_BYTES - 4096) // per_window, replace=False))
        arrays = {k: a[keep] for k, a in arrays.items()}
        arrays["window_index"] = keep.astype(np.float64)
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, f"{name}.npy"), a)


def device_view(address: int, shape, typestr: str, device: torch.device) -> torch.Tensor:
    """a tensor over a device buffer the library owns (no copy; valid as long as the library keeps the buffer)"""
    class View:
        __cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (address, False), "version": 2}

    return torch.as_tensor(View(), device=device)


# ------------------------------------------------------------------------------------ reference arm
def run_reference(args):
    """The reference's CPU path (oracle port: reference diart block logic restated in oracle/, torch-CPU
    restatement of the pyannote networks), all host threads, same workload in bounded samples."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import nets
    from oracle.pipeline import OraclePipeline

    nets.STABLE = False       # a timing leg: one evaluation per call (the reproducibility double-check is for reference VALUES)
    pipe = OraclePipeline(nets.make_segmentation(), nets.make_embedding(), as_reference=True)
    rb = args.ref_batch
    data = torch.from_numpy(make_stream_batches(0, 1, 2 * rb)[0])
    cores = pick_threads(pipe, data)
    nb = data.shape[0] // rb
    for i in range(args.warmup):
        pipe(data[(i % nb) * rb:(i % nb + 1) * rb])
    t0 = time.perf_counter()
    for i in range(args.steps):
        out = pipe(data[(i % nb) * rb:(i % nb + 1) * rb])
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        seg, emb, maps, margins = out
        dump_outputs(args.dump_outputs, {"segmentation": seg, "embeddings": emb, "speaker_map": maps, "margins": margins})
    value = args.steps * rb * STEP_SECONDS / dt
    sample = f"{args.steps} steps x {rb} consecutive windows (of the batch-256 workload), K-fold repeated trunk as the reference runs it"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample_batch": rb},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    _RESULT_LINES.append(json.dumps(line))


def pick_threads(pipe, data) -> int:
    """torch's CPU kernels do not scale to every core of a 128-core host on these layer sizes (the LSTM in
    particular gets slower); give the CPU arm the thread count that is fastest on a short, time-boxed probe."""
    cores = os.cpu_count() or 1
    best, best_t = min(16, cores), float("inf")
    t_start = time.perf_counter()
    for n in sorted({min(cores, c) for c in (16, 32, 64)}):
        torch.set_num_threads(n)
        pipe.nets(data[:4])
        t0 = time.perf_counter()
        pipe.nets(data[:8])
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = n, dt
        if time.perf_counter() - t_start > 40:           # a loaded host: stop probing, keep the best so far
            break
    torch.set_num_threads(best)
    return best


def cpu_baseline(budget_s: float = 12.0, rb: int = 32):
    from oracle import nets
    from oracle.pipeline import OraclePipeline

    pipe = OraclePipeline(nets.make_segmentation(), nets.make_embedding(), as_reference=True)
    data = torch.from_numpy(make_stream_batches(0, 1, 2 * rb)[0])
    stable, nets.STABLE = nets.STABLE, False         # a timing leg: one evaluation per call
    try:
        cores = pick_threads(pipe, data)
        pipe(data[:rb])                              # warm-up
        n, t0 = 0, time.perf_counter()
        while n < 2 or (time.perf_counter() - t0 < budget_s and n < 12):
            pipe(data[(n % 2) * rb:(n % 2 + 1) * rb])
            n += 1
        dt = time.perf_counter() - t0
    finally:
        nets.STABLE = stable
    return {"value": n * rb * STEP_SECONDS / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{n} batches x {rb} consecutive windows of the same stream, oracle pipeline (K-fold repeated "
                      f"trunk as the reference runs it), torch CPU float32, {dt:.1f} s"}


# ------------------------------------------------------------------------------------------ our arm
def run_ours(args):
    from diart_b200 import _lib, blocks, models, synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the diart_b200 path has no CPU fallback")
    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist_mod.init_process_group("nccl", device_id=device)
        dist = dist_mod
    lib = _lib.lib()
    B = args.batch
    config = blocks.SpeakerDiarizationConfig(
        segmentation=models.SegmentationModel(models.B200SegmentationLoader(synth.segmentation_state())),
        embedding=models.EmbeddingModel(models.B200EmbeddingLoader(
            synth.wespeaker_state() if args.embedding == "wespeaker" else synth.embedding_state())),
        device=device)
    pipe = blocks.SpeakerDiarization(config)
    NB = 3                                                  # 3 x 82 MB of distinct inputs > 126 MB L2
    host = make_stream_batches(rank, NB, B)
    dev = [torch.from_numpy(host[j]).to(device) for j in range(NB)]
    pinned = [torch.from_numpy(host[j]).pin_memory() for j in range(NB)]

    def barrier():
        torch.cuda.synchronize(device)
        if dist is not None:
            dist.barrier()

    # ---------------- device-resident throughput (`value`) with per-kernel CUDA-event timing
    fused, F, K, D = pipe._ensure_fused(CHUNK)
    stream = _lib.stream_ptr(device)

    shared = None
    seg_p, emb_p, map_p = C.c_void_p(), C.c_void_p(), C.c_void_p()

    def run_steps(n):
        """n pipeline steps through dg_pipeline_submit / collect: the clustering of step i overlaps the networks of steps
        i+1, i+2; every step's results are complete when the last collect is reached on the stream.  The last step's results:
        serial, the returned (segmentation, embeddings, speaker map) device tensors; pipelined, the device pointers left in
        seg_p / emb_p / map_p (the handle's slot buffers, valid until the third next submit)"""
        if args.serial:
            out = None
            for i in range(n):
                out = pipe.device_step(dev[i % NB])
            return out
        collect = lambda: _lib.check(lib.dg_pipeline_collect(fused, C.byref(seg_p), C.byref(emb_p), C.byref(map_p), stream))
        for i in range(n):           # three steps outstanding, like the host-buffer leg
            _lib.check(lib.dg_pipeline_submit(fused, dev[i % NB].data_ptr(), B, CHUNK, stream))
            if i > 1:
                collect()
        for _ in range(min(n, 2)):
            collect()

    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        run_steps(args.warmup)
        barrier()
        lib.dg_profile_enable(1)
        launches0 = lib.dg_launch_count()
        clocks.mark()
        ev0.record()
        last = run_steps(args.steps)
        ev1.record()
        torch.cuda.synchronize(device)
        lib.dg_profile_enable(0)
        launches = lib.dg_launch_count() - launches0
        if args.dump_outputs and rank == 0:      # copied before any further step reuses the slot buffers
            if last is None:
                last = (device_view(seg_p.value, (B, F, K), "<f4", device), device_view(emb_p.value, (B, K, D), "<f4", device),
                        device_view(map_p.value, (B, K), "<i4", device))
            dump_outputs(args.dump_outputs, dict(zip(("segmentation", "embeddings", "speaker_map"), (t.cpu().numpy() for t in last))))
        t_wait = time.monotonic()
        while not clocks.rows and clocks.proc is not None and time.monotonic() - t_wait < 3.0:
            run_steps(args.steps)            # nvidia-smi has not delivered a line yet: keep the same load until it does (untimed)
            torch.cuda.synchronize(device)
    ms = ev0.elapsed_time(ev1)
    buf = C.create_string_buffer(1 << 16)
    lib.dg_profile_report(buf, len(buf))
    kernels = json.loads(buf.value.decode())
    t = torch.tensor([ms], device=device, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * args.steps * B * STEP_SECONDS / (ms_max / 1e3)

    # ---------------- end to end through the C ABI with HOST buffers (H2D + D2H inside the call)
    seg_h = [torch.empty((B, F, K)).pin_memory() for _ in range(3)]
    emb_h = [torch.empty((B, K, D)).pin_memory() for _ in range(3)]
    map_h = [torch.empty((B, K), dtype=torch.int32).pin_memory() for _ in range(3)]

    def host_steps(n):
        """host buffers in, host buffers out, every step: pinned waveforms are uploaded inside submit_host, the
        step's scores / embeddings / speaker map are downloaded inside collect_host (blocking)"""
        if args.serial:
            for i in range(n):
                _lib.check(lib.dg_pipeline_step_host(fused, pinned[i % NB].data_ptr(), B, CHUNK, seg_h[0].data_ptr(),
                                                     emb_h[0].data_ptr(), map_h[0].data_ptr(), None))
            return
        depth = 3      # two steps compute, the third one's waveforms are uploaded meanwhile
        for i in range(n):
            _lib.check(lib.dg_pipeline_submit_host(fused, pinned[i % NB].data_ptr(), B, CHUNK))
            if i >= depth - 1:
                j = (i - depth + 1) % 3
                _lib.check(lib.dg_pipeline_collect_host(fused, seg_h[j].data_ptr(), emb_h[j].data_ptr(), map_h[j].data_ptr()))
        for i in range(max(0, n - depth + 1), n):
            j = i % 3
            _lib.check(lib.dg_pipeline_collect_host(fused, seg_h[j].data_ptr(), emb_h[j].data_ptr(), map_h[j].data_ptr()))

    host_steps(max(2, args.warmup))
    barrier()
    t0 = time.perf_counter()
    host_steps(args.steps)
    torch.cuda.synchronize(device)
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], device=device, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * args.steps * B * STEP_SECONDS / float(t.item())

    # ---------------- BASELINE config 5: shared speaker identity across the ranks -- after every step ONE all-gather of
    # centroid-delta records (NCCL, ~82 KB per rank) + a deterministic merge, stream-ordered on the clustering stream so that the
    # three-deep pipelining of the networks is kept (device-resident inputs, like `value`)
    ident_line = None
    if (world > 1 or args.shared_identity) and not args.serial:
        from diart_b200.parallel import SharedIdentity

        pipe.reset()
        fused, F, K, D = pipe._ensure_fused(CHUNK)
        ident = SharedIdentity(pipe.clustering)

        def ident_steps(n):          # three steps outstanding, like `value`
            for i in range(n):
                _lib.check(lib.dg_pipeline_submit(fused, dev[i % NB].data_ptr(), B, CHUNK, stream))
                ident.sync_submitted(fused)
                if i > 1:
                    _lib.check(lib.dg_pipeline_collect(fused, None, None, None, stream))
            for _ in range(min(n, 2)):
                _lib.check(lib.dg_pipeline_collect(fused, None, None, None, stream))

        ident_steps(max(2, args.warmup))
        barrier()
        lib.dg_profile_enable(1)
        i0, i1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        i0.record()
        ident_steps(args.steps)
        i1.record()
        torch.cuda.synchronize(device)
        ibuf = C.create_string_buffer(1 << 16)
        lib.dg_profile_report(ibuf, len(ibuf))
        lib.dg_profile_enable(0)
        ik = json.loads(ibuf.value.decode())
        t = torch.tensor([i0.elapsed_time(i1)], device=device, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ident_ms = float(t.item())
        ag_us = None
        if dist is not None:      # the collective alone, back to back (latency-bound: 82 KB per rank)
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            for _ in range(5):
                dist.all_gather_into_tensor(ident._gathered, ident._rec)
            a0.record()
            for _ in range(50):
                dist.all_gather_into_tensor(ident._gathered, ident._rec)
            a1.record()
            torch.cuda.synchronize(device)
            ag_us = 1e3 * a0.elapsed_time(a1) / 50
        per = lambda k: 1e3 * ik[k]["ms"] / ik[k]["count"] if k in ik else None
        ident_line = {"value": world * args.steps * B * STEP_SECONDS / (ident_ms / 1e3), "unit": UNIT,
                      "ms_per_step": ident_ms / args.steps, "allgather_us": ag_us, "merge_us": per("cluster_merge"),
                      "export_us": per("cluster_export"), "record_bytes_per_rank": int(ident._rec.numel()) * 8,
                      "protocol": "per step: export of this rank's centroid changes -> one all-gather -> merge in rank order "
                                  "(identical tables on all ranks), on the clustering stream between the clustering of step i and "
                                  "of step i+1; the networks of steps i+1, i+2 overlap it"}

    # ---------------- end to end with the ring buffer in HBM (SURVEY.md 8(f) row 3): the host pushes every sample once
    # (B x 8000 new samples per step instead of B stacked windows), windows are formed on the device
    stream_line = None
    if not args.serial and not args.no_stream_leg:
        from diart_b200 import synth as _synth
        from diart_b200.operators import DeviceAudioStream

        n_total = max(2, args.warmup) + args.steps
        audio = _synth.synth_audio(CHUNK + STEP * (n_total * B - 1), seed=1234 + rank)
        dst = DeviceAudioStream(CHUNK / SR, STEP / SR, SR, max_windows=B, device=device)
        pipe.reset()
        fused, F, K, D = pipe._ensure_fused(CHUNK)
        dst.push(audio[:CHUNK - STEP])
        cursor = [CHUNK - STEP]

        def stream_steps(n):
            depth = 3
            for i in range(n):
                blk = audio[cursor[0]:cursor[0] + B * STEP]
                cursor[0] += B * STEP
                _lib.check(lib.dg_stream_push_host(dst.handle, blk.ctypes.data, len(blk)))
                _lib.check(lib.dg_pipeline_submit_stream(fused, dst.handle, B))
                if i >= depth - 1:
                    j = (i - depth + 1) % 3
                    _lib.check(lib.dg_pipeline_collect_host(fused, seg_h[j].data_ptr(), emb_h[j].data_ptr(), map_h[j].data_ptr()))
            for i in range(max(0, n - depth + 1), n):
                j = i % 3
                _lib.check(lib.dg_pipeline_collect_host(fused, seg_h[j].data_ptr(), emb_h[j].data_ptr(), map_h[j].data_ptr()))

        stream_steps(max(2, args.warmup))
        barrier()
        t0 = time.perf_counter()
        stream_steps(args.steps)
        torch.cuda.synchronize(device)
        st_s = time.perf_counter() - t0
        t = torch.tensor([st_s], device=device, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        stream_line = {"value": world * args.steps * B * STEP_SECONDS / float(t.item()), "unit": UNIT,
                       "ms_per_step": 1e3 * float(t.item()) / args.steps, "h2d_bytes_per_step": B * STEP * 4,
                       "d2h_bytes_per_step": B * F * K * 4 + B * K * D * 4 + B * K * 4,
                       "api": "dg_stream_push_host (pageable host block -> pinned mirror -> ring in HBM) + dg_pipeline_submit_stream / "
                              "collect_host, three steps outstanding"}
        del dst

    # ---------------- R3: the drop-in call itself, SpeakerDiarization.__call__ on B separate SlidingWindowFeatures (the
    # reference's Chronometer bracket, src/diart/inference.py:130-137): gather + H2D, fused step, device post-path, D2H of
    # the turn list, Annotation objects -- everything a StreamingInference user pays per batch
    call_line = None
    if not args.no_pipeline_call:
        from diart_b200.core import SlidingWindow, SlidingWindowFeature

        pipe.reset()
        sw_of = lambda n: SlidingWindow(start=STEP_SECONDS * n, duration=1 / SR, step=1 / SR)
        rows = [[np.ascontiguousarray(host[j][b][:, None]) for b in range(B)] for j in range(NB)]
        n_calls = args.steps

        def call_steps(n, first):
            """the timed bracket is the reference's: `pipeline(batch)` only (inference.py:130-137); the batch objects exist before"""
            turns, spent = 0, 0.0
            for i in range(n):
                g0 = (first + i) * B
                chunks = [SlidingWindowFeature(rows[i % NB][b], sw_of(g0 + b)) for b in range(B)]
                t0 = time.perf_counter()
                out = pipe(chunks)
                spent += time.perf_counter() - t0
                turns += sum(len(a) for a, _ in out)
            return turns, spent

        call_steps(2, 0)
        barrier()
        pipe.call_profile = {}
        n_turn_objs, call_s = call_steps(n_calls, 2)
        prof = pipe.call_profile
        pipe.call_profile = None
        t = torch.tensor([call_s], device=device, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        call_line = {"value": world * n_calls * B * STEP_SECONDS / float(t.item()), "unit": UNIT,
                     "ms_per_call": 1e3 * float(t.item()) / n_calls, "calls": n_calls,
                     "h2d_bytes_per_step": int(lib.dg_pipeline_last_call_h2d_bytes(pipe._fused)),
                     "d2h_bytes_per_step": B * 16 + 4 + 4 * (n_turn_objs // n_calls),
                     "phases_ms_per_call": {k: round(1e3 * v / max(1, prof.get("calls", 1)), 3) for k, v in prof.items() if k != "calls"},
                     "api": "SpeakerDiarization.__call__(Sequence[SlidingWindowFeature]) -> Sequence[(Annotation, SlidingWindowFeature)], "
                            "synchronous per batch (dg_pipeline_call_host: the B separate pageable host windows are compared with "
                            "their predecessors by worker threads and, being consecutive hops of one stream, uploaded once and re-formed on "
                            "the device; pipelined sub-batches of the fused step, device aggregation/binarisation, one D2H of the turn list)"}

    # ---------------- parity of the benchmarked configuration (outside every timed region): the pipelined path over NB
    # batches of B windows from a fresh state; speaker maps against the oracle clustering replayed on the same scores /
    # embeddings, float64 centroids bit for bit, a sample of the scores against the oracle network
    parity = None
    if rank == 0 and not args.no_parity_check:
        from oracle import nets as onets
        from oracle.clustering import OracleClustering

        def measure_parity():
            pipe.reset()
            fused, F, K, D = pipe._ensure_fused(CHUNK)
            got = []
            for i in range(NB):
                pipe.submit(dev[i])
                if i > 0:
                    got.append(pipe.collect())
            got.append(pipe.collect())
            torch.cuda.synchronize(device)
            cfg = pipe.config
            replay = OracleClustering(cfg.tau_active, cfg.rho_update, cfg.delta_new, "cosine", cfg.max_speakers)
            ok, bad = True, None
            for j, (sg, em, mp) in enumerate(got):
                sg, em, mp = sg.cpu().numpy(), em.cpu().numpy(), mp.cpu().numpy()
                want = np.stack([replay(s_, e_)[0] for s_, e_ in zip(sg, em)])
                if not np.array_equal(want, mp):
                    ok, bad = False, (j, int(np.where((want != mp).any(axis=1))[0][0]))
                    break
            centers_equal = bool(ok and np.array_equal(pipe.clustering.centers, replay.centers))
            with torch.no_grad():
                torch.set_num_threads(min(16, os.cpu_count() or 1))
                o_seg = onets.make_segmentation()(torch.from_numpy(host[0][:4])[:, None, :]).numpy()
            seg_err = float(np.abs(got[0][0][:4].cpu().numpy() - o_seg).max())
            emb_err = None
            if args.embedding == "xvector":      # unit-norm embeddings of the same 4 windows against the oracle network
                from oracle.pipeline import osp_block
                with torch.no_grad():
                    o_emb = onets.make_embedding().forward_dedup(torch.from_numpy(host[0][:4])[:, None, :], osp_block(torch.from_numpy(o_seg)))
                    o_emb = (o_emb / o_emb.norm(dim=-1, keepdim=True)).numpy()
                emb_err = float(np.abs(got[0][1][:4].cpu().numpy() - o_emb).max())
            if os.environ.get("DG_BENCH_PARITY_DETAIL") == "1":      # diagnostic: which windows of which batch deviate
                with torch.no_grad():
                    net = onets.make_segmentation()
                    for j in range(NB):
                        idx = [0, 1, 2, 3, B // 2, B - 2, B - 1]
                        o = net(torch.from_numpy(host[j][idx])[:, None, :]).numpy()
                        g = got[j][0].cpu().numpy()[idx]
                        print(f"parity detail: batch {j}: per-window seg max abs err " +
                              " ".join(f"{w}:{np.abs(g[q] - o[q]).max():.1e}" for q, w in enumerate(idx)), file=sys.stderr)
            parity = {"chunks": NB * B, "maps_equal_oracle_replay": ok, "centroids_bit_equal": centers_equal,
                      "seg_max_abs_err_4_windows": seg_err, "emb_max_abs_err_4_windows": emb_err, "first_difference": bad}
            if not (ok and centers_equal and seg_err < 1e-4 and (emb_err is None or emb_err < 1e-4)):
                # which side moved?  the same batch once more, one step at a time on a fresh state, and the oracle once more
                pipe.reset()
                seg2 = pipe.device_step(dev[0])[0][:4].cpu().numpy()
                with torch.no_grad():
                    o_seg2 = onets.make_segmentation()(torch.from_numpy(host[0][:4])[:, None, :]).numpy()
                parity["diagnosis"] = {"pipelined_vs_serial_rerun": float(np.abs(got[0][0][:4].cpu().numpy() - seg2).max()),
                                       "serial_rerun_vs_oracle": float(np.abs(seg2 - o_seg).max()),
                                       "oracle_vs_oracle_rerun": float(np.abs(o_seg - o_seg2).max())}
                print(json.dumps({"parity_failed": parity}), file=sys.stderr)
                parity["failed"] = True
            return parity

        parity = measure_parity()
        if parity.get("failed"):
            # (round 2 traced three such reports to the torch CPU oracle's first float32 evaluation in a process, DESIGN.md section 4;
            # the oracle now double-checks itself.)  Measure once more; a second failure is fatal, a pass is reported together
            # with the first attempt
            first = parity
            parity = measure_parity()
            parity["first_attempt"] = first
            if parity.get("failed"):
                raise SystemExit(f"bench.py: the benchmarked configuration fails its parity check twice: {parity}")

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    # ---------------- roofline of the dominant kernel
    # `roofline` = the kernel with the largest CUDA-event time inside the timed region.  At B = 256 that is one of the two
    # sequential kernels -- cluster_step (ONE CTA on its own stream) or lstm_rec (2 x ceil(B/16) CTAs) -- which are long but narrow
    # and overlap everything else; `by_sm_time` therefore also ranks by event time x the fraction of the 148 SMs a kernel occupies,
    # and `step` puts the whole step against both rooflines.
    pk = peaks()
    narrow = {"cluster_step": 1 / 148, "cluster_merge": 1 / 148, "cluster_export": 1 / 148, "relabel_maps": 1 / 148,
              "lstm_rec": min(1.0, 2 * ((B + 15) // 16) / 148)}
    sm_time = {k: v["ms"] * narrow.get(k, 1.0) for k, v in kernels.items()}
    dom = max(kernels, key=lambda k: kernels[k]["ms"])        # the dominant kernel BY EVENT DURATION inside the timed region
    dom_sm = max(sm_time, key=sm_time.get)                     # ... and by SM-time (extra key `by_sm_time`)
    per_launch_ms = kernels[dom]["ms"] / kernels[dom]["count"]
    traffic_tab = {}
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        traffic_tab = json.load(open(tpath))
    traffic = traffic_tab.get(dom)

    def tensor_line(k):
        ms_l = kernels[k]["ms"] / kernels[k]["count"]
        if k in FLOPS_PER_CHUNK_STEP:       # several launches per step under one tag: total FLOPs of the step / total time
            tf = FLOPS_PER_CHUNK_STEP[k] * B * args.steps / (kernels[k]["ms"] * 1e-3) / 1e12
        else:
            tf = FLOPS_PER_CHUNK[k] * B / (ms_l * 1e-3) / 1e12
        return {"kernel": k, "bound": "tensor", "achieved": tf, "peak": pk["tf"], "unit": "TFLOP/s", "frac": tf / pk["tf"],
                "traffic": traffic_tab.get(k), "peak_source": pk["src"] + " (bf16 sustained)", "ms_per_launch": ms_l,
                "executed_x3": 3 * tf, "frac_of_peak_executed": 3 * tf / pk["tf"]}

    def hbm_line(k):
        ms_l = kernels[k]["ms"] / kernels[k]["count"]
        gbs = HBM_BYTES_PER_CHUNK[k] * B / (ms_l * 1e-3) / 1e9
        return {"kernel": k, "bound": "hbm", "achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gbs / pk["hbm_gbs"],
                "traffic": traffic_tab.get(k), "peak_source": pk["src"], "ms_per_launch": ms_l}

    def line_of(k):
        if k in HBM_BYTES_PER_CHUNK:
            return hbm_line(k)
        if k in FLOPS_PER_CHUNK or k in FLOPS_PER_CHUNK_STEP:
            return tensor_line(k)
        ms_l = kernels[k]["ms"] / kernels[k]["count"]
        achieved = BYTES_PER_CHUNK * B / (ms_l * 1e-3) / 1e9
        return {"kernel": k, "bound": "hbm", "achieved": achieved, "peak": pk["hbm_gbs"], "unit": "GB/s",
                "frac": achieved / pk["hbm_gbs"], "traffic": traffic_tab.get(k), "peak_source": pk["src"], "ms_per_launch": ms_l}

    roofline = line_of(dom)
    roofline["dominant_by"] = "CUDA-event duration summed over the timed region"
    if dom in ("lstm_rec", "cluster_step"):
        roofline["note"] = ("latency-bound sequential kernel (293 dependent steps per launch / one dependent step per chunk) on a few SMs, "
                            "overlapped by the wide kernels of the other streams: neither roofline binds it; see `recurrence`, `by_sm_time` and `step`")
    roofline["by_sm_time"] = dict(line_of(dom_sm), dominant_by="SM-time (event ms x SMs occupied / 148)")
    roofline["sm_time_ms_per_step"] = {k: round(v / args.steps, 4) for k, v in sorted(sm_time.items(), key=lambda kv: -kv[1])[:6]}
    if "lstm_rec" in kernels:   # the longest kernel by duration: neither roofline binds a recurrence
        r_ms = kernels["lstm_rec"]["ms"] / kernels["lstm_rec"]["count"]
        roofline["recurrence"] = {
            "kernel": "lstm_rec", "ms_per_launch": r_ms, "us_per_dependent_step": r_ms * 1e3 / 293,
            "achieved_tflops": FLOPS_PER_CHUNK["lstm_rec"] * B / (r_ms * 1e-3) / 1e12, "traffic": traffic_tab.get("lstm_rec"),
            "note": "latency-bound: 293 dependent steps per launch (4 launches = 1172 per batch), 2 x ceil(B/16) CTAs of 16 batch rows "
                    "(8 rows up to 128 windows); tcgen05 with fp16 hi/lo planes, W_hh resident in tensor memory; per step 96 MMAs "
                    "(tensor pipe ~1.1 k cycles) then a MUFU-bound cell update; cycle table in profiles/r2_lstm_step_timing.log"}
    gemms = {k: v for k, v in kernels.items() if k.startswith("tdnn") or k.startswith("resnet_l")}
    if gemms:   # the largest throughput-bound tensor kernel, for the tensor roofline proper
        gk = max(gemms, key=lambda k: gemms[k]["ms"])
        roofline["largest_gemm"] = tensor_line(gk)
    step_flops = sum(FLOPS_PER_CHUNK[k] * (4 if k == "lstm_inproj" or k == "lstm_rec" else 2 if k in
                     ("sinc0", "sinc_conv1", "sinc_conv2", "seg_linear") else 1) for k in FLOPS_PER_CHUNK) * B
    step_ms = ms_max / args.steps
    sfc = STEP_FLOPS_PER_CHUNK_WESPEAKER if args.embedding == "wespeaker" else STEP_FLOPS_PER_CHUNK
    roofline["step"] = {
        "bound": "tensor", "flops_per_step": sfc * B, "achieved": sfc * B / (step_ms * 1e-3) / 1e12,
        "peak": pk["tf"], "unit": "TFLOP/s", "frac": sfc * B / (step_ms * 1e-3) / 1e12 / pk["tf"],
        "peak_source": pk["src"] + " (bf16 sustained)", "compulsory_bytes_per_step": BYTES_PER_CHUNK * B,
        "hbm_frac": BYTES_PER_CHUNK * B / (step_ms * 1e-3) / 1e9 / pk["hbm_gbs"],
        "traffic": traffic_tab.get("_step"),
        "note": "SURVEY.md 8(d) algorithmic FLOPs of the de-duplicated path (3.359 GFLOP per chunk) / ms_per_step; the path executes 3 "
                "tcgen05 products per algorithmic product (fp16 hi/lo split) and contains 1172 + 256 dependent steps per batch"}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD if args.embedding == "xvector" else WORKLOAD.replace(
                       "pyannote/embedding architectures", "pyannote/wespeaker-voxceleb-resnet34-LM (variant B) architectures"),
                   "embedding": args.embedding, "batch": B, "streams": world, "parallelism": (f"{world} independent streams, "
                   "1 per GPU, no collectives" if shared is None else f"{world} streams, 1 per GPU, shared speaker "
                   "identity: one NCCL all-gather of centroid-delta records per step + deterministic merge"), "l2": "inputs rotate over 3 distinct 82 MB batches (246 MB > 126 MB L2)",
                   "arithmetic": "float32 results: every dense layer as fp16 hi/lo operand planes x 3 tcgen05 products with float32 "
                                 "accumulation (22 significand bits per operand), float64 clustering"},
        "chunks_per_s": value / STEP_SECONDS,
        "step_tflops": step_flops / (ms_max / args.steps * 1e-3) / 1e12,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": B * CHUNK * 4,
                "d2h_bytes_per_step": B * F * K * 4 + B * K * D * 4 + B * K * 4,
                "api": ("dg_pipeline_step_host" if args.serial else "dg_pipeline_submit_host / collect_host, three steps outstanding") +
                       " (C ABI, pinned host buffers)"},
        "shared_identity": ident_line,
        "e2e_stream": stream_line,
        "e2e_pipeline_call": call_line,
        "parity": parity,
        "gpu_launches": int(launches),
        "clocks": clocks.summary(),
        "roofline": roofline,
        "kernels_ms_per_step": {k: round(v["ms"] / args.steps, 4) for k, v in sorted(kernels.items(),
                                                                                     key=lambda kv: -kv[1]["ms"])},
    }
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline()
    _RESULT_LINES.append(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def main():
    # the driver parses ONE JSON line from stdout: anything libraries print (e.g. NCCL's version banner) goes to
    # stderr instead; the real stdout is restored only for the result line
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        _main()
    finally:
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        os.close(real_stdout)
    for line in _RESULT_LINES:
        print(line, flush=True)


_RESULT_LINES = []


def _main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)       # 20 steps = 65 ms of device time; the whole default run takes about a minute
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--ref-batch", type=int, default=32)
    ap.add_argument("--embedding", default="xvector", choices=["xvector", "wespeaker"],
                    help="embedding network: pyannote/embedding (XVectorSincNet, the quoted configuration) or variant B, "
                         "pyannote/wespeaker-voxceleb-resnet34-LM (ResNet34, reference README.md:172-173)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-stream-leg", action="store_true", help="skip the device ring-buffer leg (e2e_stream)")
    ap.add_argument("--no-pipeline-call", action="store_true", help="skip the SpeakerDiarization.__call__ leg (e2e_pipeline_call)")
    ap.add_argument("--no-parity-check", action="store_true", help="skip the oracle replay of the benchmarked configuration")
    ap.add_argument("--shared-identity", action="store_true",
                    help="BASELINE config 5: share the global speaker table across ranks (one all-gather per step)")
    ap.add_argument("--serial", action="store_true", help="one step at a time (dg_pipeline_step) instead of depth-2 pipelining")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step (segmentation, embeddings, speaker map) as DIR/<name>.npy; "
                         "the inputs are seeded, so runs with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
