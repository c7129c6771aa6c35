#!/usr/bin/env python
"""Benchmark of the H.264 intra reconstruction hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--frames F] [--distinct G] [--rgb-scale S] [--e2e-frames E] [--pipeline fused|split]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of F synthetic 1920x1088 High-profile IDR pictures
(BASELINE.json configs[2]) that are already resident in HBM: ONE launch of the fused kernel kf_recon
(dequantisation + inverse transforms + intra prediction + residual add + RGB24, see DESIGN.md), or with
--pipeline split round 1's kernels 1, 2, 3.  Rank 0 prints ONE JSON line.  Multi-GPU: one process per GPU
(torchrun), disjoint pictures per GPU, no collective on the data path ("scaling": "weak").

What the line carries besides `value` (device-timed, resident inputs):
  e2e          the same through the C ABI with HOST buffers (mvg_decode_host_packed: pinned packed SoA in, RGB24 out);
               scope: after the CAVLC parse (the boundary of SURVEY.md section 8b)
  stream_e2e   Annex-B bytes in host memory -> host front end (CAVLC on the host cores) -> C ABI -> RGB24 in host
               memory, on EVERY rank, summed: the like-for-like figure beside the reference arm, which also parses
  configs3     BASELINE.json configs[3]: 8000 pictures sharded over the GPUs, RGB thumbnails at 1/4 size
  split_pipeline  round 1's three kernels on the same batch (kept for one round for comparison)
  parity_checked  pictures of every timed path were downloaded after the timed region and compared (SHA-256) with
               the CPU oracle; any mismatch makes the run exit non-zero without a line

--impl reference times the reference's own CPU implementation (oracle/_ref, the unmodified reference compiled by
oracle/Makefile): one process pinned to each host core, every process decodes --ref-pics pictures.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "1080p_idr_frames_per_s_recon_rgb"
UNIT = "frames/s"
WORKLOAD = "configs[2]: 1920x1080 High-profile CAVLC, 8x8 transform + custom scaling lists, 1000 IDR frames on 1 B200"
# identical in both arms (the driver compares the dicts)
CONFIG = {"workload": WORKLOAD, "coded_size": "1920x1088", "profile": "High (100), CAVLC, transform_8x8_mode, 8 SPS scaling lists",
          "macroblock_mix": "1/3 Intra4x4, 1/3 Intra8x8, 1/3 Intra16x16", "output": "RGB24 1920x1088 (mb_to_rgb)",
          "stream": "synthetic, committed generator (minivideo_b200/csrc/h264_synth.c), seed 0xC0FFEE+2"}


# ----------------------------------------------------------------------------
# helpers

def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def sha(a) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU; result(t0, t1) keeps the samples taken
    inside the timed region [t0, t1] (time.perf_counter())."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples = index, threading.Event(), []
        self.max_mhz, self.err = None, None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons",
                                  getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons", None))
            while not self.stop_flag.is_set():
                mask = get_reasons(h) if get_reasons else 0
                self.samples.append((time.perf_counter(), nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM), mask))
                time.sleep(0.004)
        except Exception as e:  # pragma: no cover - depends on the box
            self.err = repr(e)

    def result(self, t0: float, t1: float):
        self.stop_flag.set()
        self.join(timeout=2)
        names = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "sw_power_cap": 0x4, "hw_power_brake_slowdown": 0x80}
        inside = [s for s in self.samples if t0 <= s[0] <= t1] or self.samples[-3:]
        if not inside:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "error": self.err}
        mask = 0
        for s in inside:
            mask |= s[2]
        return {"sm_mhz": float(np.median([s[1] for s in inside])), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(k for k, bit in names.items() if mask & bit), "samples": len(inside)}


def algorithmic_bytes(n_mb: int, width: int, height: int, scale: int):
    """Per picture.  SURVEY.md section 8(d) with the side information this repository actually carries
    (21 B of SoA per macroblock in, a 16-byte control record between kernels 1 and 2; the survey budgeted 32 B)."""
    meta_in = 21                      # mb_kind, i16_mode, chroma_mode, qp_y, cbp, 16 luma modes
    rgb = 3 * (width // scale) * (height // scale) if scale >= 1 else 0
    yuv = width * height * 3 // 2
    return {
        "k1": n_mb * (768 + meta_in) + n_mb * (768 + 16),
        "k2": n_mb * (768 + 16) + yuv,
        "k3": yuv + rgb,
        "kf_rgb": n_mb * (768 + meta_in) + rgb,       # fused, SoA in -> RGB24 out: what kf_recon<RGB> must move
        "kf_tiles": n_mb * (768 + meta_in) + yuv,     # fused, SoA in -> reconstructed picture out
        "kf_thumbs": n_mb * (768 + meta_in) + rgb,    # fused, SoA in -> RGB24 thumbnails out (kf_recon's thumbnail mode)
        # SURVEY.md 8(d): "if K1 is fused into K2 the algorithmic figure is N_mb*800 + 1.5WH + B_K3"
        "survey_fused_pipeline": n_mb * 800 + yuv + yuv + rgb,
    }


# ----------------------------------------------------------------------------
# reference arm: the unmodified reference decoder on the host cores

def _pinned_run(cmd, cwd, core):
    def pin():
        try:
            os.sched_setaffinity(0, {core})
        except OSError:
            pass
    return subprocess.run(cmd, capture_output=True, text=True, cwd=cwd, preexec_fn=pin)


def reference_sample(stream_path: str, cwd: str, cores: list, pics_per_proc: int, rgb: bool = True):
    """One process of the reference per host core, each pinned to its core (BASELINE.md section 3) and decoding the
    same `pics_per_proc` 1080p pictures (CAVLC parse + reconstruction + mb_to_rgb, no file output).  Returns
    (frames_per_s over the slowest process's in-process minivideo_decode() time, wall_s)."""
    import re
    from oracle import ref
    cmd = [str(ref.REF_DECODE), stream_path, str(pics_per_proc), "--time"] + ([] if rgb else ["--norgb"])
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=len(cores)) as ex:
        res = list(ex.map(lambda c: _pinned_run(cmd, cwd, c), cores))
    wall = time.perf_counter() - t0
    secs = []
    for r in res:
        m = re.search(r"REFTIME pictures=(\d+) seconds=([0-9.]+)", r.stdout)
        if r.returncode != 0 or not m or int(m.group(1)) != pics_per_proc:
            raise RuntimeError(f"ref_decode --time failed: {r.stdout[-500:]} {r.stderr[-500:]}")
        secs.append(float(m.group(2)))
    return len(cores) * pics_per_proc / max(secs), wall


class ReferenceRunner:
    """The stream the reference decodes (written once to /dev/shm) and the cores it may use."""

    def __init__(self, pics: int):
        from minivideo_b200 import synth
        from oracle import ref
        if not ref.available():
            raise RuntimeError("oracle/_ref/ref_decode is missing (run `make -C oracle ref` where the reference is mounted)")
        self.pics = pics
        self.cores = sorted(os.sched_getaffinity(0)) or [0]
        base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
        self.tmp = tempfile.TemporaryDirectory(dir=base, prefix="mvbench_")
        stream, _ = synth.generate(pics, "1080p", want_soa=False, seed=0xC0FFEE + 2)
        self.path = os.path.join(self.tmp.name, "sample.264")
        Path(self.path).write_bytes(stream)
        _pinned_run([str(ref.REF_DECODE), self.path, "1", "--time"], self.tmp.name, self.cores[0])      # page cache, binary

    def sample(self):
        return reference_sample(self.path, self.tmp.name, self.cores, self.pics)

    @property
    def description(self):
        return (f"{self.pics} pictures per process x {len(self.cores)} processes, one pinned to each host core, same 1080p "
                "stream, the unmodified reference's parse + reconstruction + mb_to_rgb (in-process minivideo_decode() time, "
                "slowest process)")


def run_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return 0
    runner = ReferenceRunner(args.ref_pics)
    vals, walls = [], []
    for i in range(args.warmup + args.steps):
        fps, wall = runner.sample()
        if i >= args.warmup:
            vals.append(fps); walls.append(wall)
    value = float(np.mean(vals))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(np.mean(walls)) * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": CONFIG,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": len(runner.cores), "kind": "reference", "sample": runner.description},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ----------------------------------------------------------------------------
# our arm

class ParityError(RuntimeError):
    pass


def run_ours(args):
    rank, world, local = dist_env()
    if args.gpus > 1 and world == 1:
        # not launched by torchrun: re-exec under it (one process per GPU)
        port = 29500 + (os.getpid() % 1000)
        os.execvp(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                                   f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
                                   "--master-port", str(port), str(Path(__file__).resolve())] + sys.argv[1:])
    import ctypes as C
    import torch
    import torch.distributed as dist
    from minivideo_b200 import api, front, synth
    from oracle import cpu          # the checker (outside every timed region)

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    try:        # run this rank (and allocate its pinned buffers) on the host cores next to its GPU
        import pynvml as nv
        nv.nvmlInit()
        nv.nvmlDeviceSetCpuAffinity(nv.nvmlDeviceGetHandleByIndex(local))
    except Exception:
        pass
    if world > 1:
        # NCCL prints its version banner on stdout at communicator creation; stdout carries the one JSON line only
        sys.stdout.flush()
        keep = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(keep, 1)
            os.close(keep)
    # the host cores are shared by the ranks: each takes its share for the bitstream path
    host_threads = args.stream_threads or max(1, (len(os.sched_getaffinity(0)) or 1) // world)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    checks = []             # (what, ok)

    def check(what, got, want):
        ok = sha(np.asarray(got).reshape(-1)) == sha(np.asarray(want).reshape(-1))
        checks.append((what, ok))
        if not ok:
            raise ParityError(f"rank {rank}: {what} differs from the oracle")

    # ---- synthetic input: G distinct pictures per rank, replicated on the device to F
    F, G, scale = args.frames, min(args.distinct, args.frames), args.rgb_scale
    P3 = 8000 // max(world, 2) if args.configs3 else 0          # configs[3]: 8000 pictures over 2/4/8 GPUs
    _, soa = synth.generate(G, "1080p", want_stream=False, seed=0xC0FFEE + 2 + 1000 * rank)
    W, H, N = soa.width, soa.height, soa.n_mbs
    slots = max(F, P3)
    ctx = api.Context(local, soa.width_mbs, soa.height_mbs, slots)
    ctx.set_sps_from(soa)
    ctx.upload(soa, 0)
    for s in range(G, slots):
        ctx.clone_slot(s % G, s)
    ctx.sync()
    # what the oracle says about two of the distinct pictures (computed before anything is timed)
    probe = [0, G - 1] if G > 1 else [0]
    want_yuv = {i: cpu.reconstruct(soa.pictures(i, 1))[0][0] for i in probe}

    def oracle_rgb(i, s):
        return cpu.yuv_to_rgb(want_yuv[i][None], W, H, s)[0]
    want_rgb_s = {i: oracle_rgb(i, scale) for i in probe}

    # ---- timed region: K steps over the resident batch
    split = args.pipeline == "split"

    def timed_resident(n_pics, rgb_scale, use_split):
        ctx.set_pipeline_mode(api.PIPELINE_SPLIT if use_split else api.PIPELINE_FUSED)
        if use_split:
            step = lambda: ctx.run(0, n_pics, rgb_scale)            # kernels 1, 2, 3
        elif rgb_scale == 1:
            step = lambda: ctx.run_rgb(0, n_pics)                   # ONE launch: levels -> RGB24
        else:
            step = lambda: ctx.run_thumbs(0, n_pics, rgb_scale)     # ONE launch for 2, 4, 8, 16: levels -> RGB24 thumbnails
        for _ in range(args.warmup):
            step()
        ctx.sync()
        barrier()
        k_ms = {"k1": [], "k2": [], "k3": [], "kf": []}
        launches = 0
        t0 = time.perf_counter()
        ctx.mark(0)
        for _ in range(args.steps):
            step()
            t = ctx.timing()                      # waits for the step; per-kernel CUDA-event times
            k_ms["k1"].append(t.k1_dequant_idct_ms); k_ms["k2"].append(t.k2_wavefront_ms); k_ms["k3"].append(t.k3_rgb_ms)
            k_ms["kf"].append(t.fused_ms)
            launches += t.launches
        ctx.mark(1)
        dev_ms = ctx.mark_elapsed_ms()
        barrier()
        t1 = time.perf_counter()
        return dev_ms, {k: float(np.mean(v)) for k, v in k_ms.items() if np.mean(v) > 0}, launches, t0, t1

    sampler = ClockSampler(local)
    sampler.start()
    t_wait = time.perf_counter()
    while not sampler.samples and sampler.err is None and time.perf_counter() - t_wait < 10.0:
        time.sleep(0.01)                      # NVML initialisation can take longer than the warm-up
    dev_ms, mean_ms, launches, t_wall0, t_wall1 = timed_resident(F, scale, split)
    wall_ms = (t_wall1 - t_wall0) * 1e3
    clocks = sampler.result(t_wall0, t_wall1)
    dump = None
    if args.dump_outputs and rank == 0:
        # the RGB24 pictures the last timed step left in HBM, before the other pipeline overwrites them; F full pictures
        # are gigabytes, so a fixed seeded sample: every eighth row (seeded choice) of eight pictures (seeded choice)
        rng = np.random.default_rng(0xC0FFEE)
        dump_slots = np.sort(rng.choice(F, min(F, 8), replace=False))
        dump_rows = np.sort(rng.choice(H // scale, max(1, H // scale // 8), replace=False))
        dump = {"rgb": np.stack([ctx.download_rgb(int(s), scale)[dump_rows] for s in dump_slots]).astype(np.float32),
                "rgb_slots": dump_slots.astype(np.float64), "rgb_rows": dump_rows.astype(np.float64)}
    # what was timed produced the right pictures: a source slot, a clone in the middle, one of the last slots
    for s in sorted({probe[-1], (F // 2) // G * G + probe[0] if F >= 2 * G else probe[0], (F - 1) // G * G + probe[0] if F > G else probe[0]}):
        if s < F:
            check(f"resident RGB, slot {s}", ctx.download_rgb(s, scale), want_rgb_s[s % G])

    # the other pipeline on the same batch, for comparison (round 1's three kernels / the fused kernel)
    other_dev_ms, other_ms, other_launches, _, _ = timed_resident(F, scale, not split)
    check("resident RGB (other pipeline)", ctx.download_rgb(probe[0], scale), want_rgb_s[probe[0]])
    ctx.set_pipeline_mode(api.PIPELINE_SPLIT if split else api.PIPELINE_FUSED)

    # ---- configs[3]: 8000 pictures sharded over the GPUs, RGB thumbnails at 1/4 size (resident + end to end)
    configs3 = None
    if P3:
        c3_dev_ms, c3_ms, c3_launches, _, _ = timed_resident(P3, 4, split)
        check("configs[3] RGB at 1/4 size", ctx.download_rgb((P3 - 1) // G * G + probe[0] if P3 > G else probe[0], 4), oracle_rgb(probe[0], 4))
        launches += c3_launches
        configs3 = {"dev_ms": c3_dev_ms, "kernels_ms": c3_ms}

    # ---- end to end: pinned host buffers -> H2D -> kernels -> D2H RGB in pinned host memory, through the
    # C ABI.  Headline: the packed transfer format (mvg_decode_host_packed, what the front end emits);
    # the dense SoA call (mvg_decode_host) is timed beside it.
    E = min(args.e2e_frames, F)
    rgb_px = (W // scale) * (H // scale) * 3
    rgb_out = api.PinnedArray((E, rgb_px), np.uint8)
    d2h = rgb_out.nbytes
    packed = api.Packed(soa, n_pics=E, pinned=True)
    h2d = packed.nbytes

    def timed_host(fn):
        for _ in range(max(1, args.warmup // 2)):
            fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    def timed_host_two_in_flight(outs, rgb_scale, pk):
        """The asynchronous form of the same call (mvg_submit_packed / mvg_wait, what INTEGRATION.md's binding does): step k + 1
        is submitted before step k is waited for, into the other output buffer, so that the copy engines do not drain
        between steps.  Every step still copies its inputs host -> device and its result device -> host."""
        def run(n):
            tk = api.submit_packed(ctx, pk, None, outs[0].array, rgb_scale)
            for i in range(1, n):
                t2 = api.submit_packed(ctx, pk, None, outs[i & 1].array, rgb_scale)
                ctx.wait(tk)
                tk = t2
            ctx.wait(tk)
        run(max(2, args.warmup // 2))
        barrier()
        t0 = time.perf_counter()
        run(args.steps)
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    rgb_out.array[...] = 0
    e2e_blocking_s = timed_host(lambda: ctx.decode_host_packed(packed, None, rgb_out.array, scale))
    for k in sorted({probe[-1], (E - 1) // G * G + probe[0] if E > G else probe[0]}):
        if k < E:
            check(f"end-to-end RGB, picture {k}", rgb_out.array[k], want_rgb_s[k % G])
    rgb_out2 = api.PinnedArray((E, rgb_px), np.uint8)
    rgb_out.array[...] = 0
    rgb_out2.array[...] = 0
    e2e_s = timed_host_two_in_flight([rgb_out, rgb_out2], scale, packed)
    for name, buf in (("first", rgb_out), ("second", rgb_out2)):
        check(f"end-to-end RGB, two submissions in flight, {name} buffer", buf.array[probe[-1]], want_rgb_s[probe[-1] % G])
    del rgb_out2

    reps = -(-E // G)
    pin = {
        "mb_kind": api.PinnedArray((E * N,), np.uint8), "i16_mode": api.PinnedArray((E * N,), np.uint8),
        "chroma_mode": api.PinnedArray((E * N,), np.uint8), "qp_y": api.PinnedArray((E * N,), np.int8),
        "cbp": api.PinnedArray((E * N,), np.uint8), "luma_modes": api.PinnedArray((E * N, 16), np.uint8),
        "coeff": api.PinnedArray((E * N, 384), np.int16),
    }
    for name, pa in pin.items():
        src = getattr(soa, name)
        pa.array[...] = np.concatenate([src] * reps)[: E * N]
    batch = api.Batch()
    batch.n_pics = E
    for name, pa in pin.items():
        setattr(batch, name, pa.ptr)
    h2d_dense = sum(pa.nbytes for pa in pin.values())
    rgb_out.array[...] = 0
    e2e_dense_s = timed_host(lambda: ctx.decode_host(None, None, rgb_out.array, scale, batch=batch))
    check("end-to-end RGB (dense levels)", rgb_out.array[probe[-1]], want_rgb_s[probe[-1]])
    del pin, batch

    c3_e2e_s = None
    if P3:
        E3 = min(E, P3)
        out4 = api.PinnedArray((E3, (W // 4) * (H // 4) * 3), np.uint8)
        packed3 = packed if E3 == E else api.Packed(soa, n_pics=E3, pinned=True)
        out4b = api.PinnedArray((E3, (W // 4) * (H // 4) * 3), np.uint8)
        c3_blocking_s = timed_host(lambda: ctx.decode_host_packed(packed3, None, out4.array, 4))
        c3_e2e_s = timed_host_two_in_flight([out4, out4b], 4, packed3)
        check("configs[3] end-to-end RGB at 1/4 size", out4.array[probe[0]], oracle_rgb(probe[0], 4))
        check("configs[3] end-to-end RGB at 1/4 size, second buffer", out4b.array[probe[0]], oracle_rgb(probe[0], 4))
        configs3.update(e2e_s=c3_e2e_s, e2e_blocking_s=c3_blocking_s, e2e_pictures=E3, d2h=out4.nbytes)
        del out4, out4b, packed3
    del packed

    # ---- from the bitstream, on every rank: Annex-B bytes -> host front end (CAVLC on this rank's share of the host
    # cores, a persistent parser, packed output into pinned memory) -> mvg_decode_host_packed -> RGB24 in pinned host
    # memory.  Same input and output as the reference arm.  A step = S pictures in sub-batches of B: the parse of
    # sub-batch k+1 overlaps the GPU work of sub-batch k (what mvt_extract() does with its two buffer sets).
    stream_e2e = None
    stream_s, S = 0.0, 0
    if args.stream_frames > 0:
        S, B = args.stream_frames, min(args.stream_batch, args.stream_frames)
        D = min(S, 64)                                          # distinct pictures in the stream, visited cyclically
        stream, _ = synth.generate(D, "1080p", want_soa=False, seed=0xC0FFEE + 2 + 1000 * rank)
        st = front.Stream(stream)
        info = st.info
        ls4, ls8 = st.level_scale()
        ctx.set_sps(info.width_mbs, info.height_mbs, ls4, ls8, info.cb_qp_offset, info.cr_qp_offset)
        flib = front.lib()
        parser = C.c_void_p()
        if flib.mvf_parser_create(st.handle, host_threads, C.byref(parser)) != 1:
            raise RuntimeError("mvf_parser_create failed")
        order = ("mb_kind", "i16_mode", "chroma_mode", "qp_y", "luma_modes", "nz_blocks", "word_off", "pic_off", "words")
        idx_all = np.ascontiguousarray(np.arange(S, dtype=np.int32) % D)

        def buffers(cap):
            pk = {"mb_kind": api.PinnedArray((B * N,), np.uint8), "i16_mode": api.PinnedArray((B * N,), np.uint8),
                  "chroma_mode": api.PinnedArray((B * N,), np.uint8), "qp_y": api.PinnedArray((B * N,), np.int8),
                  "luma_modes": api.PinnedArray((B * N, 16), np.uint8), "nz_blocks": api.PinnedArray((B * N,), np.uint32),
                  "word_off": api.PinnedArray((B * N,), np.uint32), "pic_off": api.PinnedArray((B + 1,), np.uint64),
                  "words": api.PinnedArray((cap,), np.uint16)}
            return pk, front.FrontPackedBatch(B, *(pk[k].ptr for k in order), cap), api.PackedBatch(B, *(pk[k].ptr for k in order))
        # right-sized pinned buffers: a first parse into a token buffer fails on capacity and reports what a sub-batch needs
        probe_set = buffers(1)
        flib.mvf_parser_parse_packed(parser, idx_all.ctypes.data, 0, B, C.byref(probe_set[1]))
        cap = int(probe_set[1].words_needed * 1.25) + 4096
        del probe_set
        sets = [buffers(cap), buffers(cap)]
        outs = [api.PinnedArray((B, rgb_px), np.uint8), api.PinnedArray((B, rgb_px), np.uint8)]
        n_sub = -(-S // B)

        def parse(k):
            cnt = min(B, S - k * B)
            rc = flib.mvf_parser_parse_packed(parser, idx_all[k * B:].ctypes.data, 0, cnt, C.byref(sets[k & 1][1]))
            if rc != 1:
                raise RuntimeError(flib.mvf_parser_last_error(parser).decode())
            return cnt

        def decode(k, cnt):
            sets[k & 1][2].n_pics = cnt
            ctx._ck(ctx.lib.mvg_decode_host_packed(ctx.handle, C.byref(sets[k & 1][2]), None, outs[k & 1].ptr, scale))

        def stream_step(ex):
            cnt = parse(0)
            for k in range(n_sub):
                nxt = ex.submit(parse, k + 1) if k + 1 < n_sub else None
                decode(k, cnt)
                if nxt:
                    cnt = nxt.result()
        with ThreadPoolExecutor(max_workers=1) as ex:           # ctypes calls release the GIL
            stream_step(ex)                                     # warm-up
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                stream_step(ex)
            torch.cuda.synchronize()
            stream_s = time.perf_counter() - t0
        # the last sub-batch is still in its output buffer: one of its pictures against the oracle, from the stream
        k_last = n_sub - 1
        dense = st.parse(indices=[int(idx_all[k_last * B])], n_threads=1)
        o_sps = cpu.OracleSps()
        o_sps.width_mbs, o_sps.height_mbs = info.width_mbs, info.height_mbs
        C.memmove(o_sps.ls4, np.ascontiguousarray(ls4, np.int32).ctypes.data, 288 * 4)
        C.memmove(o_sps.ls8, np.ascontiguousarray(ls8, np.int32).ctypes.data, 384 * 4)
        o_sps.cb_qp_offset, o_sps.cr_qp_offset = info.cb_qp_offset, info.cr_qp_offset
        yuv1 = np.zeros(W * H * 3 // 2, np.uint8)
        arrs = [np.ascontiguousarray(x) for x in (dense.mb_kind, dense.i16_mode, dense.chroma_mode, dense.qp_y, dense.luma_modes, dense.coeff)]
        pv = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
        cpu.lib().oracle_reconstruct_picture(C.byref(o_sps), *[pv(a) for a in arrs], pv(yuv1[:W * H]), pv(yuv1[W * H:W * H * 5 // 4]),
                                             pv(yuv1[W * H * 5 // 4:]), None)
        check("bitstream-to-RGB, last sub-batch", outs[k_last & 1].array[0], cpu.yuv_to_rgb(yuv1[None], W, H, scale)[0])
        flib.mvf_parser_destroy(parser)
        stream_e2e = {"pictures_per_step_per_gpu": S, "sub_batch": B, "host_threads_per_gpu": host_threads,
                      "stream_bytes_per_picture": len(stream) // D, "distinct_pictures": D,
                      "pinned_words_per_sub_batch": cap}
        del sets, outs

    # ---- reduce over ranks (max time), rank 0 reports
    times = torch.tensor([dev_ms, wall_ms, e2e_s * 1e3, e2e_dense_s * 1e3, stream_s * 1e3, other_dev_ms,
                          configs3["dev_ms"] if configs3 else 0.0, (c3_e2e_s or 0.0) * 1e3, e2e_blocking_s * 1e3,
                          (configs3["e2e_blocking_s"] if configs3 else 0.0) * 1e3], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    (dev_ms, wall_ms, e2e_ms, e2e_dense_ms, stream_ms, other_dev_ms, c3_dev_ms, c3_e2e_ms, e2e_blocking_ms,
     c3_blocking_ms) = (float(x) for x in times.tolist())

    if rank == 0:
        peak, peak_src = measured_peak()
        ab = algorithmic_bytes(N, W, H, scale)
        name_of = {"k1": "k1_dequant_idct", "k2": "k2_wavefront", "k3": "k3_rgb", "kf": "kf_recon"}
        ab_of = dict(ab, kf=ab["kf_rgb"] if scale == 1 else ab["kf_thumbs"] if scale in (2, 4, 8, 16) else ab["kf_tiles"])
        dom = max(mean_ms, key=mean_ms.get)
        achieved = ab_of[dom] * F / (mean_ms[dom] * 1e-3) / 1e9
        traffic = None
        tfile = ROOT / "profiles" / "ncu_traffic.json"
        if tfile.exists():
            try:
                traffic = json.loads(tfile.read_text())["per_picture_dram_bytes"][dom] * F
            except Exception:
                traffic = None

        def kernel_block(ms):
            return {name_of[k]: {"ms_per_launch": v, "algorithmic_bytes": ab_of[k] * F, "achieved_gbs": ab_of[k] * F / (v * 1e-3) / 1e9,
                                 "frac": ab_of[k] * F / (v * 1e-3) / 1e9 / peak} for k, v in ms.items()}
        step_ms = dev_ms / args.steps
        line = {
            "metric": METRIC, "value": world * F * args.steps / (dev_ms * 1e-3), "unit": UNIT,
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": CONFIG,
            "run": {"pictures_per_step_per_gpu": F, "distinct_pictures": G, "rgb_scale": scale,
                    "pipeline": "split: k1_dequant_idct, k2_wavefront -> tiles, k3_rgb" if split else
                                "fused: one launch of kf_recon per step (levels in HBM -> RGB24 in HBM)",
                    "l2": f"inputs {F * N * 789 / 1e9:.1f} GB per step >> 126 MB L2 (no flush needed)",
                    "timing": "CUDA events on the launch stream, max over ranks", "wall_ms_per_step": wall_ms / args.steps},
            "clocks": clocks,
            "e2e": {"value": world * E * args.steps / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "pictures_per_step_per_gpu": E,
                    "scope": "post-parse: starts from the parsed structure-of-arrays (the C-ABI boundary, SURVEY.md 8b); the "
                             "reference arm also parses -- stream_e2e is the like-for-like figure",
                    "path": "mvg_submit_packed / mvg_wait, two steps in flight (step k + 1 submitted before step k is waited for, two "
                            "output buffers): pinned host packed SoA (sparse levels) -> H2D -> k0 expand, kf_recon -> D2H RGB24",
                    "blocking": {"value": world * E * args.steps / (e2e_blocking_ms * 1e-3),
                                 "path": "mvg_decode_host_packed, one call per step: the copy engines drain between steps"},
                    "dense": {"value": world * E * args.steps / (e2e_dense_ms * 1e-3), "h2d_bytes_per_step": h2d_dense,
                              "path": "mvg_decode_host: dense int16[384] levels per macroblock"}},
            "gpu_launches": launches,
            # SURVEY.md 8(d) is the contract for `achieved`: algorithmic bytes per picture x pictures per launch / launch time.
            # For the fused pipeline the survey's figure is N_mb*800 + 1.5WH + B_K3 = 19 061 760 B at scale 1 (it still counts
            # a tiles round trip and kernel 3's traffic, which kf_recon<RGB> no longer has); `roofline_actual_bytes` below is
            # the same launch against what the kernel really has to move (SoA in, RGB24 out).
            "roofline": ({"bound": "hbm", "kernel": "kf_recon", "achieved": ab["survey_fused_pipeline"] * F / (mean_ms["kf"] * 1e-3) / 1e9,
                          "peak": peak, "unit": "GB/s", "frac": ab["survey_fused_pipeline"] * F / (mean_ms["kf"] * 1e-3) / 1e9 / peak,
                          "traffic": traffic, "peak_source": peak_src,
                          "algorithmic_bytes_per_picture": ab["survey_fused_pipeline"],
                          "basis": "SURVEY.md 8(d), k1 fused into k2: N_mb*800 + 1.5*W*H + (1.5 + 3)*W*H",
                          "note": "kf_recon is bound by the shared-memory/LSU data pipe (81 % of its peak) and instruction issue (81 % issue-active), "
                                  "not by HBM: profiles/r02_final_kf_rgb_summary.txt, profiles/r02_notes.md"}
                         if dom == "kf" and scale == 1 else
                         {"bound": "hbm", "kernel": name_of[dom], "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                          "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_picture": ab_of[dom]}),
            "roofline_actual_bytes": {"kernel": name_of[dom], "algorithmic_bytes_per_picture": ab_of[dom],
                                      "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                                      "note": "what the dominant kernel itself has to move per picture (kf_recon<RGB>: 789 B of SoA per "
                                              "macroblock in, RGB24 out; no residual, no tiles)"},
            "kernels": kernel_block(mean_ms),
            ("fused_pipeline" if split else "split_pipeline"): {
                "value": world * F * args.steps / (other_dev_ms * 1e-3), "ms_per_step": other_dev_ms / args.steps,
                "kernels": kernel_block(other_ms), "launches": other_launches,
                "roofline_all_stages": {"frac": sum(ab_of[k] for k in other_ms) * F / (sum(other_ms.values()) * 1e-3) / 1e9 / peak}},
            "parity_checked": bool(checks) and all(ok for _, ok in checks),
            "parity_checks": [w for w, _ in checks],
        }
        if stream_e2e:
            stream_e2e.update(value=world * S * args.steps / (stream_ms * 1e-3), unit=UNIT,
                              path="Annex-B bytes -> mvf_parser_parse_packed (CAVLC on the host cores, persistent workers) -> "
                                   "mvg_decode_host_packed -> RGB24; sub-batch k+1 is parsed while sub-batch k is on the GPU; "
                                   "every rank runs its own feeder on its share of the host cores, the value is the sum")
            line["stream_e2e"] = stream_e2e
        if configs3:
            ab3 = algorithmic_bytes(N, W, H, 4)
            line["configs3"] = {
                "workload": "configs[3]: 1920x1080 High-profile batch of 8000 IDR frames sharded across 2/4/8 B200 with fused RGB thumbnail downscale",
                "pictures_per_gpu": P3, "pictures_total": P3 * world, "rgb_scale": 4,
                "value": world * P3 * args.steps / (c3_dev_ms * 1e-3), "unit": UNIT, "ms_per_step": c3_dev_ms / args.steps,
                "kernels_ms": configs3["kernels_ms"],
                "pipeline": ("k1, k2 -> macroblock tiles, k3_rgb_scaled (1/4 size box average)" if split else
                             "one launch of kf_recon in thumbnail mode per step (levels in HBM -> RGB24 at 1/4 size in HBM)"),
                "algorithmic_bytes_per_picture": (ab3["kf_tiles"] + ab3["k3"]) if split else ab3["kf_thumbs"],
                "e2e": {"value": world * configs3["e2e_pictures"] * args.steps / (c3_e2e_ms * 1e-3), "unit": UNIT,
                        "pictures_per_step_per_gpu": configs3["e2e_pictures"], "d2h_bytes_per_step": configs3["d2h"], "h2d_bytes_per_step": h2d,
                        "scope": "post-parse (mvg_submit_packed / mvg_wait, two steps in flight), RGB24 at 480x272 back to pinned host memory",
                        "blocking": world * configs3["e2e_pictures"] * args.steps / (c3_blocking_ms * 1e-3)},
                "note": "at 1 GPU the batch is 4000 pictures (half of configs[3], which names 2/4/8 GPUs)" if world == 1 else None}
        if world == 1 and not args.no_cpu_baseline:
            try:
                runner = ReferenceRunner(args.ref_pics)
                fps, _ = runner.sample()
                line["cpu_baseline"] = {"value": fps, "unit": UNIT, "cores": len(runner.cores), "kind": "reference", "sample": runner.description}
                if stream_e2e:
                    line["stream_e2e"]["vs_cpu_baseline"] = stream_e2e["value"] / fps
            except Exception as e:
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": f"unavailable: {e}"}
        print(json.dumps(line), flush=True)
    if dump is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dump.items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), a)
    ctx.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=1000, help="pictures per step per GPU (resident in HBM)")
    ap.add_argument("--distinct", type=int, default=32, help="distinct pictures generated on the host per GPU")
    ap.add_argument("--rgb-scale", type=int, default=1, help="RGB thumbnail downscale factor (1 = the reference's mb_to_rgb)")
    ap.add_argument("--e2e-frames", type=int, default=384, help="pictures per end-to-end step per GPU")
    ap.add_argument("--stream-frames", type=int, default=1024, help="pictures per step of the bitstream-to-RGB measurement (0 = skip)")
    ap.add_argument("--stream-batch", type=int, default=128, help="pictures per sub-batch of the bitstream-to-RGB measurement")
    ap.add_argument("--stream-threads", type=int, default=0, help="parser threads per GPU (0 = this rank's share of the host cores)")
    ap.add_argument("--ref-pics", type=int, default=30, help="pictures each host core decodes in the CPU baseline / reference arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs3", dest="configs3", action="store_false", help="skip the configs[3] block (8000 pictures, 1/4-size RGB)")
    ap.add_argument("--pipeline", default="fused", choices=["fused", "split"], help="fused kernel (default) or round 1's three kernels")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a seeded sample of the RGB24 output of the last step as float32 DIR/rgb.npy "
                         "(rank 0; picture slots and rows in DIR/rgb_slots.npy, DIR/rgb_rows.npy); "
                         "--impl reference writes nothing")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)
    try:
        return run_ours(args)
    except ParityError as e:
        print(f"bench.py: PARITY FAILURE: {e}", file=sys.stderr, flush=True)
        return 3


if __name__ == "__main__":
    sys.exit(main())
