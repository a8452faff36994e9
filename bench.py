#!/usr/bin/env python
"""bench.py -- encode/decode GSamples/s of the FLAC hot path on B200 (driver contract).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload c3|c5|c4] [--dump-outputs DIR]

Workload (default c3 = BASELINE.json configs[2], the configuration the encode-scaling metric is
quoted on; it fits one GPU): synthetic Sentinel-2-like 10980x10980 uint16, 8 bands, streaming
tile_size 1024 -> 121 tiles / 964 483 200 samples, compression level 5.  A "step" is one pass of
the encode hot path over that raster, resident in HBM: per-tile min/max -> normalise -> subframe
analysis + Rice coding -> frame assembly (+ the size read-back that fixes the byte offsets).
After the K timed encode steps the decode direction (sync scan -> Rice decode/LPC restore ->
CRC-16 -> denormalise) is timed the same way and reported under "decode".

N > 1 is STRONG scaling of that ONE scene (north_star: "work is sharded across the GPUs of one box
by tile"): one process per GPU, rank r holds and codes the contiguous row-major block of tiles
distributed.tile_shards gives it (balanced by pixel count: 15-17 of the 121 tiles at N = 8), the per-tile sizes are
all-gathered over NCCL (the one collective; its scan gives the container's byte offsets) and
`value` = the scene's samples / the slowest rank's time.  After the timed regions the ranks write
ONE container with distributed.write_sharded_container and rank 0 re-reads its index and decodes
tiles of three different ranks through the public SpatialFLACStreamer as a check (at N = 1 it also
reads the whole scene back with get_tiles_by_bbox: "container_check.bbox_all").  The old weak
number (every rank codes a whole scene) is kept under "weak".  "cpu_baseline.ffmpeg" holds the
second labelled CPU row: FFmpeg libavcodec's FLAC encoder and decoder on one core.

`e2e` is the same step through the public engine API with HOST (pinned) buffers: H2D of the
raster and D2H of the frames inside the timed region.  "c5_bbox" is BASELINE.json configs[4]
through the public API: SpatialFLACStreamer.get_tiles_by_bbox over a 4096-tile container, the
requested tiles split over the ranks.  Every timed section runs K steps after its warm-up.

`--dump-outputs DIR` writes what the last timed encode and decode steps returned as DIR/<name>.npy (float32 / float64,
the frame bytes and the decoded raster as a fixed seeded sample of 2^22 elements each, under 64 MB in all); the inputs
are synthetic and seeded, so two builds run with the same arguments can be compared array for array.

`--impl reference` times the reference's CPU implementation of the path (the oracle port of
libFLAC's procedure + the reference's numpy normalisation, one tile per task in a process pool over
all host cores, windows read from a file and tile FLACs written to files as cli.py:553-622 does)
on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import sys
import tempfile
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "encode GSamples/s (streaming tiles -> FLAC frames; decode GSamples/s reported beside it)"
UNIT = "GSamples/s"

WORKLOADS = {
    # name: (description, level, tile_size, bands)
    "c3": ("synthetic Sentinel-2-like 10980x10980 uint16 x 8 bands, streaming tile_size 1024 (121 tiles), level 5", 5, 1024, 8),
    "c5": ("4096 tiles of 512x512 int16 (batch decode sweep corpus), level 5", 5, 512, 1),
    "c4": ("synthetic float32 DEM 32768x32768 via normalize_to_audio, level 8, single stream", 8, 32768, 1),
}

# modelled integer operations per sample (SURVEY.md 8d) for the issue-rate roofline, and the measured integer issue
# peak of this pool's B200 (profiles/r01_int_peak_b200.txt: adds / IADD3+IMAD mixes reach 3.86-3.89 warp instructions
# per clock and SM = 36 T lane-ops/s; a pure shift/logic stream half of that)
MODEL_OPS = {"decode": 25.0, "encode_l5": 70.0, "encode_l8": 300.0}
INT_PEAK_TOPS = 36.2


def scene_shape(workload: str, scale_div: int = 1):
    if workload == "c3":
        s = 10980 // scale_div
        return 8, s, s
    if workload == "c5":
        return 1, (4096 // (scale_div * scale_div)) * 512, 512
    s = 32768 // scale_div
    return 1, s, s


def make_rows(workload: str, device, r0: int, r1: int, scale_div: int = 1):
    """Rows [r0, r1) of the workload's scene as a (bands, r1-r0, W) tensor (same values as the full raster)."""
    from flac_raster_b200 import synth
    nb, H, W = scene_shape(workload, scale_div)
    if workload == "c3":
        return synth.sentinel2_like(r1 - r0, W, 8, device=device, row0=r0)
    if workload == "c5":
        assert r0 % 512 == 0 and r1 % 512 == 0
        return synth.dem_int16_tiles((r1 - r0) // 512, 512, device=device, first_tile=r0 // 512)
    assert r0 == 0 and r1 == H
    return synth.dem_float32(H, W, device=device)


class ClockSampler(threading.Thread):
    """Samples SM clocks and throttle reasons during the timed region (NVML every 4 ms, nvidia-smi as fallback)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._halt = threading.Event()

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self._nvml_index())
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            bits = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
            get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
            while not self._halt.is_set():
                try:
                    self.samples.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                    r = int(get_reasons(h))
                    for n, b in bits.items():
                        if r & int(b):
                            self.reasons.add(n)
                except Exception:  # noqa: BLE001
                    pass
                self._halt.wait(0.004)
            return
        except Exception:  # noqa: BLE001
            pass
        import subprocess
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip().splitlines()
                if out:
                    f = [x.strip() for x in out[0].split(",")]
                    self.samples.append(float(f[0]))
                    self.max_mhz = float(f[1])
                    for n, v in zip(names, f[2:6]):
                        if v.lower().startswith("active"):
                            self.reasons.add(n)
            except Exception:  # noqa: BLE001
                pass
            self._halt.wait(0.2)

    def _nvml_index(self) -> int:
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        try:
            ids = [int(v) for v in vis.split(",") if v.strip() != ""]
            if ids and self.index < len(ids):
                return ids[self.index]
        except ValueError:
            pass
        return self.index

    def stop(self):
        self._halt.set()
        self.join(timeout=6)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ----------------------------------------------------------------------------- CPU reference arm
# The reference's per-tile path (cli.py:558-598 -> converter.py:99-154): read the window from a file, interleave,
# normalize_to_audio (numpy), libFLAC-procedure encode (oracle C port), write the tile's FLAC file; decode: read that
# file, decode, denormalize_from_audio.  One tile per task; tasks run in a process pool (BASELINE.md section 3).
def cpu_tile_encode(args):
    npy, r0, r1, c0, c1, level, out_path = args
    from oracle import flac_oracle as fo, normalization_oracle as no
    arr = np.load(npy, mmap_mode="r")
    win = np.ascontiguousarray(arr[:, r0:r1, c0:c1])
    bands, h, w = win.shape
    inter = win.transpose(1, 2, 0).reshape(-1, bands)
    rate, bits = no.calculate_audio_params((h, w), win.dtype)
    audio, prm = no.normalize_to_audio(inter, bits)
    enc, _ = fo.encode(audio, 16 if bits == 16 else 32, rate, level)
    with open(out_path, "wb") as fh:
        fh.write(enc)
    return inter.size, len(enc), str(win.dtype), prm["data_min"], prm["data_max"], prm["scale_factor"]


def cpu_tile_decode(args):
    path, dtype, dmin, dmax, scale = args
    from oracle import flac_oracle as fo, normalization_oracle as no
    with open(path, "rb") as fh:
        enc = fh.read()
    pcm, _ = fo.decode(enc)
    a = pcm.astype(np.int16) if scale == 32767 else pcm
    out = no.denormalize_from_audio(a, dmin, dmax, dtype, scale)
    return int(out.size)


def _cpu_worker_init():
    from oracle import flac_oracle as fo
    fo.lib()


def sample_geometry(workload: str, n_tiles: int):
    """Windows of the first n_tiles tiles (row-major) of the workload and the rows of the scene they need."""
    desc, level, tile, bands = WORKLOADS[workload]
    if workload == "c3":
        per_row = (10980 + tile - 1) // tile
        rows = min(10980, ((n_tiles + per_row - 1) // per_row) * tile)
        wins = []
        for i in range(n_tiles):
            ty, tx = divmod(i, per_row)
            wins.append((ty * tile, min(rows, (ty + 1) * tile), tx * tile, min(10980, (tx + 1) * tile)))
        return wins, rows, level
    if workload == "c5":
        return [(i * 512, (i + 1) * 512, 0, 512) for i in range(n_tiles)], n_tiles * 512, level
    side = 2048                     # CPU sample of the float32 DEM: top-left crops of the same formula
    return [(i * side, (i + 1) * side, 0, side) for i in range(n_tiles)], n_tiles * side, level


class CpuArm:
    """Bounded sample of the workload on the host cores; keeps one process pool for all repetitions."""

    def __init__(self, workload: str, n_tiles: int, procs: int, device):
        from flac_raster_b200 import synth
        self.workload, self.procs = workload, procs
        self.wins, rows, self.level = sample_geometry(workload, n_tiles)
        base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
        self.dir = tempfile.mkdtemp(prefix="frb_cpu_", dir=base)
        if workload == "c3":
            r = synth.sentinel2_like(rows, 10980, 8, device=device)
        elif workload == "c5":
            r = synth.dem_int16_tiles(n_tiles, 512, device=device)
        else:
            r = synth.dem_float32(rows, 2048, device=device)
        arr = r.cpu().numpy()
        self.npy = os.path.join(self.dir, "scene.npy")
        np.save(self.npy, arr)                               # the "TIFF" every task reads its window from
        del r, arr
        self.pool = None
        if procs > 1:
            import multiprocessing as mp
            self.pool = mp.get_context("spawn").Pool(procs, initializer=_cpu_worker_init)
            self.pool.map(abs, range(procs))                 # workers up before anything is timed
        else:
            _cpu_worker_init()

    def run(self):
        """One pass: (encode GS/s, decode GS/s, samples)."""
        ejobs = [(self.npy, r0, r1, c0, c1, self.level, os.path.join(self.dir, f"tile_{i}.flac")) for i, (r0, r1, c0, c1) in enumerate(self.wins)]
        t0 = time.perf_counter()
        res = self.pool.map(cpu_tile_encode, ejobs, chunksize=1) if self.pool else [cpu_tile_encode(j) for j in ejobs]
        te = time.perf_counter() - t0
        samples = sum(r[0] for r in res)
        djobs = [(j[6], r[2], r[3], r[4], r[5]) for j, r in zip(ejobs, res)]
        t0 = time.perf_counter()
        got = self.pool.map(cpu_tile_decode, djobs, chunksize=1) if self.pool else [cpu_tile_decode(j) for j in djobs]
        td = time.perf_counter() - t0
        assert sum(got) == samples
        self.comp_bytes = sum(r[1] for r in res)
        return samples / te / 1e9, samples / td / 1e9, samples

    def describe(self, samples):
        return (f"first {len(self.wins)} tiles of the workload ({samples} samples), oracle C port of libFLAC 1.4.3's procedure + numpy "
                f"normalisation, one tile per task, {'process pool of ' + str(self.procs) if self.procs > 1 else 'one process'}; windows read "
                f"from a file, tile FLACs written to and read from files (cli.py:553-622)")

    def close(self):
        if self.pool:
            self.pool.close()
            self.pool.join()
        shutil.rmtree(self.dir, ignore_errors=True)


def ffmpeg_decode_baseline(workload: str, n_tiles: int, device):
    """Second, labelled CPU row: FFmpeg 8 libavcodec's FLAC decoder (a production SIMD codec, the only one on the box;
    BASELINE.md 3.2b) on GPU-made tile files of the workload, one thread.  Returns a dict or None."""
    try:
        from oracle import ffmpeg_flac as ff
        if not ff.available():
            return None
        from flac_raster_b200 import flacfmt
        from flac_raster_b200.engine import default_engine, tile_grid
        wins, rows, level = sample_geometry(workload, n_tiles)
        nb, H, W = scene_shape(workload)
        r = make_rows(workload, device, 0, rows) if workload != "c4" else None
        if r is None:
            return None
        tiles = tile_grid(r.shape[1], r.shape[2], WORKLOADS[workload][2])[:n_tiles]
        enc = default_engine().encode_tiles(r, tiles, level)
        payload = enc.payload.cpu().numpy()
        d = tempfile.mkdtemp(prefix="frb_ff_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
        try:
            paths = []
            for i in range(len(tiles)):
                si = flacfmt.StreamInfo(4096, 4096, 0, 0, int(enc.sample_rates[i]), nb, enc.bps, int(enc.n_samples[i]))
                p = os.path.join(d, f"t{i}.flac")
                with open(p, "wb") as fh:
                    fh.write(flacfmt.build_header(si))
                    fh.write(payload[int(enc.offsets[i]):int(enc.offsets[i] + enc.sizes[i])].tobytes())
                paths.append(p)
            t0 = time.perf_counter()
            n = 0
            for p in paths:
                n += ff.decode_file(p, nb).size
            dt = time.perf_counter() - t0
            # libavcodec's FLAC ENCODER over the same tiles (decoded AVFrames fed back in; only the encoder is timed)
            enc_value, enc_note = None, ""
            try:
                te, ne, be = 0.0, 0, 0
                for p in paths:
                    sec, ns, nbytes = ff.encode_timing(p, level, 4096)
                    te += sec; ne += ns * nb; be += nbytes
                enc_value = ne / te / 1e9
                enc_note = f"; encode: libavcodec flac encoder, compression_level {level}, frame_size 4096, {be} bytes out vs {int(enc.sizes.sum())} from the GPU encoder"
            except Exception as ex:  # noqa: BLE001
                enc_note = f"; encode failed: {ex!r}"
        finally:
            shutil.rmtree(d, ignore_errors=True)
        return {"decode_value": n / dt / 1e9, "encode_value": enc_value, "unit": UNIT, "cores": 1, "kind": "ffmpeg-libavcodec (not libFLAC)",
                "sample": f"first {len(tiles)} tiles ({n} samples), FLAC codec only (no (de)normalise, no file write), frames made by the GPU encoder" + enc_note}
    except Exception as ex:  # noqa: BLE001
        return {"decode_value": None, "encode_value": None, "kind": "ffmpeg-libavcodec (not libFLAC)", "sample": f"failed: {ex!r}"}


_REAL_STDOUT = None


def emit_line(obj):
    """The ONE JSON line of the contract, on the process's real stdout."""
    data = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, data)
    else:
        sys.stdout.write(data.decode())
        sys.stdout.flush()


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def run_reference(args, rank):
    if rank != 0:
        return 0
    import torch
    desc, level, tile_size, bands = WORKLOADS[args.workload]
    dev = torch.device("cuda", 0) if torch.cuda.is_available() else torch.device("cpu")
    cores = host_cores()
    n_tiles = args.cpu_tiles or max(2 * cores, 8)
    arm = CpuArm(args.workload, n_tiles, cores, dev)
    try:
        for _ in range(max(0, min(args.warmup, 1))):
            arm.run()
        vals = []
        t_all = time.perf_counter()
        for _ in range(args.steps):
            e, d, samples = arm.run()
            vals.append((e, d))
        ms = (time.perf_counter() - t_all) / max(args.steps, 1) * 1e3
        sdesc = arm.describe(samples)
    finally:
        arm.close()
    e = float(np.median([v[0] for v in vals]))
    d = float(np.median([v[1] for v in vals]))
    emit_line({
        "impl": "reference", "metric": METRIC, "value": e, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "int32", "data": "synthetic",
        "config": {"workload": desc, "level": level, "tile_size": tile_size, "blocksize": 4096},
        "decode": {"value": d, "unit": UNIT},
        "cpu_baseline": {"value": e, "unit": UNIT, "cores": cores, "kind": "port", "sample": sdesc, "decode_value": d},
        "e2e": {"value": e, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })
    return 0


def main():
    # Libraries (NCCL's version banner, torch warnings) sometimes write to fd 1: route everything except the
    # final JSON line to stderr so stdout carries exactly one line.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=list(WORKLOADS))
    ap.add_argument("--scale-div", type=int, default=1, help="shrink the workload (debug only; invalid as a result)")
    ap.add_argument("--cpu-tiles", type=int, default=0, help="tiles in the CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the weak-scaling, container and c5_bbox sections")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last encode and decode step returned as DIR/<name>.npy (float32/float64; "
                         "payload bytes and raster pixels as a fixed seeded sample; rank 0's tiles when there are several ranks)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank)
    return run_ours(args, rank, world, local)


def run_ours(args, rank, world, local):
    import torch
    import torch.distributed as dist

    from flac_raster_b200 import _native as nat
    from flac_raster_b200.distributed import (SizeExchange, allgather_tile_sizes, bind_to_gpu_numa_node, exclusive_scan, init_from_env,
                                              shard_plan, tile_shards)
    from flac_raster_b200.engine import Engine, tile_grid

    desc, level, tile_size, bands = WORKLOADS[args.workload]
    nat.require_cuda()
    numa_node = None
    if world > 1:
        numa_node = bind_to_gpu_numa_node(local)            # before any pinned allocation (first touch)
        print(f"[bench] rank {rank}: bound to NUMA node {numa_node}", file=sys.stderr)
        init_from_env("nccl")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    eng = Engine(dev)
    L = nat.lib()
    L.frb_profile_enable(1)

    # ---- the ONE scene, sharded by tile (c4 is a single stream: every rank codes all of it, i.e. replicas) ----------
    nb, H, W = scene_shape(args.workload, args.scale_div)
    ts = tile_size // (args.scale_div if args.workload != "c5" else 1)
    if args.workload == "c4":
        ts = max(H, W)
    shardable = args.workload != "c4"
    srank, sworld = (rank, world) if shardable else (0, 1)
    tiles_all, (ta, tb), (r0, r1) = shard_plan(H, W, ts, srank, sworld)
    raster = make_rows(args.workload, dev, r0, r1, args.scale_div)          # this rank's rows of the scene, resident in HBM
    tiles = tiles_all[ta:tb].copy()
    tiles["row_off"] -= r0
    n_tiles_local = len(tiles)
    samples_local = int((tiles["h"].astype(np.int64) * tiles["w"]).sum()) * nb
    samples_scene = nb * H * W if shardable else nb * H * W * world
    torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    state = {}

    # the one collective of the path: every tile's frame bytes -> global byte offsets of the container (cli.py:615-621); it is
    # enqueued on the stream inside the step and its result comes back with the step's own size download
    shards = tile_shards(tiles_all, world)
    xchg = SizeExchange(len(tiles_all), rank, world, dev, ranges=shards) if world > 1 and shardable else None

    def encode_step():
        enc = eng.encode_tiles(raster, tiles, level, size_exchange=xchg)
        if xchg is not None:
            state["offsets_all"] = exclusive_scan(enc.sizes_all)
        state["enc"] = enc
        return enc

    for _ in range(args.warmup):
        encode_step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = L.frb_launch_count()
    enc_prof, dec_prof = {}, {}

    def prof(acc, slots):
        """Device time of the library's bracketed kernels for the step that just ran (CUDA events on its stream)."""
        for name, which in slots.items():
            ms = nat.C.c_float(0)
            if L.frb_profile_last_ms(which, nat.C.byref(ms)) == 0:
                acc.setdefault(name, []).append(ms.value)

    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_wall = time.perf_counter()
    ev0.record()
    for _ in range(args.steps):
        encode_step()
        prof(enc_prof, {"k_enc_code": 0, "k_enc_stats": 4, "k_emit_frames": 2, "subframe_analysis_total": 6})
    ev1.record()
    barrier()
    enc_wall_ms = (time.perf_counter() - t_wall) * 1e3 / args.steps
    launches = L.frb_launch_count() - launches0
    enc_ms = ev0.elapsed_time(ev1) / args.steps
    enc = state["enc"]
    comp_bytes = int(enc.sizes.sum())
    dump = encode_outputs(enc) if args.dump_outputs and rank == 0 else None

    # ---- decode direction ------------------------------------------------------------------
    payload = torch.cat([enc.payload, torch.zeros(64, dtype=torch.uint8, device=dev)])
    out = torch.zeros(raster.numel() * raster.element_size(), dtype=torch.uint8, device=dev).view(raster.dtype).reshape(raster.shape)
    scale = 32767.0 if enc.bits_per_sample == 16 else 8388607.0

    def decode_step(index=enc.index()):
        # frames -> raster in one fused launch (Rice decode + predictor restore + denormalise, CRC-16 beside it); the status
        # read-back is part of the step.  Streams written by this engine carry their seek index (frame sizes + subframe bit
        # offsets, the "frbI" block of the container): no sync scan, no walk for subframe starts.  index=None is the path
        # for foreign streams (reference / libFLAC files): sync scan + skim CTAs inside the launch.
        return eng.decode_tiles(payload, enc.offsets, enc.sizes, tiles, enc.sample_rates, enc.minmax, scale, out, enc.bps, enc.blocksize,
                                index=index)

    for _ in range(max(1, args.warmup)):           # at least one: its status and raster are checked below
        st = decode_step(None)
    assert list(st[:3]) == [0, 0, 0], f"decode status {st}"
    foreign_ok = all(bool(torch.equal(out[:, int(t["row_off"]):int(t["row_off"] + t["h"]), int(t["col_off"]):int(t["col_off"] + t["w"])],
                                      raster[:, int(t["row_off"]):int(t["row_off"] + t["h"]), int(t["col_off"]):int(t["col_off"] + t["w"])]))
                     for t in tiles) if enc.bits_per_sample == 16 else None
    barrier()
    evf0, evf1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    evf0.record()
    for _ in range(args.steps):
        decode_step(None)
        prof(dec_prof, {"k_decode_subframes_scan_path": 1, "k_sync_scan": 3})
    evf1.record()
    barrier()
    dec_foreign_ms = evf0.elapsed_time(evf1) / args.steps
    out.zero_()
    for _ in range(max(1, args.warmup)):
        st = decode_step()
    assert list(st[:3]) == [0, 0, 0], f"decode status {st}"
    if enc.bits_per_sample == 16:
        # pixel for pixel inside this rank's tiles (its slab also holds rows of neighbouring ranks' tiles, which stay zero in `out`)
        lossless = all(bool(torch.equal(out[:, int(t["row_off"]):int(t["row_off"] + t["h"]), int(t["col_off"]):int(t["col_off"] + t["w"])].view(torch.int16),
                                        raster[:, int(t["row_off"]):int(t["row_off"] + t["h"]), int(t["col_off"]):int(t["col_off"] + t["w"])].view(torch.int16)))
                       for t in tiles)
    else:
        # 32-bps streams (float32 / int32 rasters quantised to 24 bits, SURVEY Q4): lossless means the decoded samples equal
        # the normalised samples that went into the encoder, compared on the device
        audio_ref, _, npx, _, _ = eng.normalize_tiles(raster, tiles)
        total = int(npx.sum()) * nb
        ref = audio_ref[:total * 4].view(torch.int32).clone()
        audio, _, st32 = eng.decode_streams(payload, enc.offsets, enc.sizes, enc.n_samples, enc.sample_rates, nb, enc.bps, enc.blocksize)
        lossless = bool(list(st32[:3]) == [0, 0, 0] and torch.equal(audio[:total * 4].view(torch.int32), ref))
        del ref
    barrier()
    dlaunch0 = L.frb_launch_count()
    ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev2.record()
    for _ in range(args.steps):
        st = decode_step()
        prof(dec_prof, {"k_decode_subframes": 1})
    ev3.record()
    barrier()
    dec_launches = L.frb_launch_count() - dlaunch0
    dec_ms = ev2.elapsed_time(ev3) / args.steps
    if dump is not None:
        dump.update(decode_outputs(out, st))
        write_outputs(args.dump_outputs, dump)
    clocks = sampler.stop() if rank == 0 else None

    # ---- e2e: host (pinned) raster in, host frames out -----------------------------------------
    host_in = torch.empty(raster.numel() * raster.element_size(), dtype=torch.uint8).pin_memory()
    host_in.copy_(raster.reshape(-1).view(torch.uint8))
    host_raster = host_in.view(raster.dtype).reshape(raster.shape)
    host_out = torch.empty(comp_bytes + (1 << 20), dtype=torch.uint8).pin_memory()

    def e2e_step():
        # public engine call with HOST buffers: H2D of every tile row, encode, D2H of the frames (pipelined inside), then the
        # size all-gather that fixes the container offsets
        e = eng.encode_tiles_host(host_raster, tiles, level, host_out=host_out)
        if world > 1 and shardable:
            allgather_tile_sizes(e.sizes, len(tiles_all), rank, world, device=dev, ranges=shards)
        return int(e.payload.numel())

    for _ in range(min(args.warmup, 2)):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    ev4, ev5 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev4.record()
    e2e_steps = args.steps
    for _ in range(e2e_steps):
        nout = e2e_step()
    ev5.record()
    barrier()
    e2e_ms = max(ev4.elapsed_time(ev5), (time.perf_counter() - t0) * 1e3) / e2e_steps

    # ---- decode e2e: host (pinned) frames in, host raster out ---------------------------------------
    host_payload = torch.empty(comp_bytes, dtype=torch.uint8).pin_memory()
    host_payload.copy_(enc.payload[:comp_bytes])
    host_back = torch.empty(raster.numel() * raster.element_size(), dtype=torch.uint8).pin_memory().view(raster.dtype).reshape(raster.shape)

    def dec_e2e_step():
        return eng.decode_tiles_host(host_payload, enc.offsets, enc.sizes, tiles, enc.sample_rates, enc.minmax, scale, host_back,
                                     enc.bps, enc.blocksize, index=enc.index())

    dec_e2e_ms = None
    if nb != 2:
        for _ in range(min(args.warmup, 2)):
            dec_e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            dst_ = dec_e2e_step()
        torch.cuda.synchronize()
        dec_e2e_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
        assert list(dst_[:3]) == [0, 0, 0], dst_
        barrier()
    del host_back, host_payload

    # ---- one container from all ranks + public-API read-back (untimed check of the sharded path) -------------------
    container = None
    if shardable and not args.no_extras:
        try:
            container = container_check(args, eng, rank, world, dev, host_raster, r0, (nb, H, W), ts, level, tiles_all)
        except Exception as ex:  # noqa: BLE001
            container = {"ok": False, "error": repr(ex)}
    del host_in, host_raster, host_out

    # ---- weak scaling (secondary): every rank codes a WHOLE scene -------------------------------------------------
    weak = None
    if world > 1 and shardable and not args.no_extras:
        full = make_rows(args.workload, dev, 0, H, args.scale_div)
        tiles_full = tile_grid(H, W, ts)
        for _ in range(2):
            eng.encode_tiles(full, tiles_full, level)
        barrier()
        evw0, evw1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        evw0.record()
        wsteps = args.steps
        for _ in range(wsteps):
            eng.encode_tiles(full, tiles_full, level)
        evw1.record()
        barrier()
        weak = evw0.elapsed_time(evw1) / wsteps
        del full

    # ---- BASELINE config 5 through the public API (4096-tile container, get_tiles_by_bbox, tiles split over the ranks) ----
    c5 = None
    if args.workload == "c3" and args.scale_div == 1 and not args.no_extras:
        del raster, out, payload
        eng.release()
        torch.cuda.empty_cache()
        try:
            c5 = c5_bbox_sweep(eng, rank, world, dev, barrier, reps=args.steps)
        except Exception as ex:  # noqa: BLE001
            c5 = {"error": repr(ex)}

    # ---- reduce over ranks (max time) -------------------------------------------------------------
    t = torch.tensor([enc_ms, dec_ms, e2e_ms, dec_e2e_ms or 0.0, weak or 0.0, enc_wall_ms,
                      (c5 or {}).get("ms", 0.0) or 0.0, dec_foreign_ms], dtype=torch.float64, device=dev)
    tot = torch.tensor([float(samples_local), float(launches), float(comp_bytes), float(nout)], dtype=torch.float64, device=dev)
    tmin = torch.cat([t, torch.tensor([1.0 if lossless else 0.0], dtype=torch.float64, device=dev)])
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    lossless = bool(float(tmin[-1]) == 1.0)                 # every rank's tiles
    enc_ms, dec_ms, e2e_ms, dec_e2e_ms, weak_ms, enc_wall_ms, c5_ms, dec_foreign_ms = (float(v) for v in t.cpu())
    enc_ms_min = float(tmin[0])
    total_samples = float(tot[0])
    comp_total, nout_total = int(tot[2]), int(tot[3])
    assert not shardable or int(total_samples) == samples_scene, (total_samples, samples_scene)
    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return 0

    peaks = {}
    pk = ROOT / "MEASURED_PEAKS.json"
    if pk.exists():
        peaks = json.loads(pk.read_text())
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"

    traffic = {}
    tf = ROOT / "profiles" / "traffic.json"          # dram__bytes_read+write per launch from the committed ncu --set full captures
    if tf.exists():
        traffic = json.loads(tf.read_text()).get(args.workload, {})
    full_launch = world == 1 and args.scale_div == 1   # the ncu traffic figures are per launch over the whole scene

    def roof(kernel_ms_list, alg_bytes, kernel, note, ops_per_sample):
        if not kernel_ms_list:
            return None
        kms = float(np.mean(kernel_ms_list))
        ach = alg_bytes / (kms * 1e-3) / 1e9
        extra = {k[len(kernel) + 1:]: v for k, v in traffic.items() if k.startswith(kernel + ":")} if full_launch else {}
        issue_ach = ops_per_sample * samples_local / (kms * 1e-3) / 1e12
        hbm_frac, issue_frac = ach / hbm_peak, issue_ach / INT_PEAK_TOPS
        return {"bound": "issue" if issue_frac >= hbm_frac else "hbm", "kernel": kernel, "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                "frac": hbm_frac, "traffic": traffic.get(kernel) if full_launch else None, "kernel_ms": kms, **extra,
                "algorithmic_bytes_per_launch": alg_bytes, "peak_source": peak_src,
                "issue": {"model_ops_per_sample": ops_per_sample, "achieved_tops": issue_ach, "peak_tops": INT_PEAK_TOPS, "frac": issue_frac,
                          "peak_source": "measured integer issue rate, profiles/r01_int_peak_b200.txt (IADD3+IMAD mix)"},
                "frac_of_slower_bound": max(hbm_frac, issue_frac), "note": note}

    def mean_ms(acc):
        return {k: float(np.mean(v)) for k, v in acc.items()}

    audio_bytes = 2 if (enc.bps == 16 and raster_elem_size(args.workload) <= 2) else 4    # planar audio element the encode kernels read (Engine.audio_elem_bytes)
    enc_alg = samples_local * audio_bytes + comp_bytes           # audio read + compressed bytes produced (SURVEY 8d)
    fused_dec = enc.bps == 16 and raster_elem_size(args.workload) <= 2 and nb != 2
    # compressed bytes consumed + output written: pixels of the raster (fused launch) or int32 audio (two-step path)
    dec_alg = comp_bytes + samples_local * (raster_elem_size(args.workload) if fused_dec else 4)
    cpu = None
    if not args.no_cpu_baseline and world == 1:      # the CPU baseline is reported by the single-GPU run only
        try:
            n_cpu = args.cpu_tiles or (8 if args.workload == "c3" else 64 if args.workload == "c5" else 4)
            arm = CpuArm(args.workload, n_cpu, 1, dev)
            try:
                ce, cd, ns = arm.run()
                cpu = {"value": ce, "unit": UNIT, "cores": 1, "kind": "port", "sample": arm.describe(ns), "decode_value": cd}
            finally:
                arm.close()
            cpu["ffmpeg"] = ffmpeg_decode_baseline(args.workload, n_cpu, dev)
        except Exception as ex:  # noqa: BLE001
            cpu = {"value": None, "unit": UNIT, "cores": 1, "kind": "port", "sample": f"failed: {ex!r}"}

    line = {
        "metric": METRIC, "value": total_samples / (enc_ms * 1e-3) / 1e9, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": enc_ms, "higher_is_better": True, "scaling": "strong" if shardable else "weak",
        "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": desc if args.scale_div == 1 else desc + f" [DEBUG scale-div {args.scale_div}]", "level": level,
                   "tile_size": ts, "blocksize": 4096, "tiles_total": len(tiles_all), "tiles_rank0": n_tiles_local,
                   "samples_total": int(total_samples), "samples_rank0": samples_local,
                   "l2": f"every rank's inputs per step ({samples_local * raster_elem_size(args.workload) / 1e6:.0f} MB of raster on rank 0) exceed the 126 MB L2; no flush needed",
                   "parallelism": (f"ONE scene, tiles sharded over {world} GPU(s) in contiguous row-major blocks, one process per GPU; "
                                   "all-gather of per-tile sizes only") if shardable else f"single stream: {world} replica(s)",
                   "numa_bound_rank0": numa_node},
        "compressed_bytes_total": comp_total, "bits_per_sample_out": comp_total * 8 / total_samples,
        "lossless_roundtrip_checked": lossless,
        "rank_ms": {"encode_max": enc_ms, "encode_min": enc_ms_min, "encode_wall_max": enc_wall_ms},
        "decode": {"value": total_samples / (dec_ms * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": dec_ms,
                   "gpu_launches": int(dec_launches),
                   "path": "streams of this engine: seek index from the container (frame sizes + subframe bit offsets), no sync scan, no skim",
                   "foreign_streams": {"value": total_samples / (dec_foreign_ms * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": dec_foreign_ms,
                                       "lossless": foreign_ok,
                                       "path": "no index (reference / libFLAC-made files): sync scan + skim CTAs that walk the Rice codes for the subframe starts"},
                   "e2e": ({"value": total_samples / (dec_e2e_ms * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": dec_e2e_ms,
                            "h2d_bytes_per_step": comp_total, "d2h_bytes_per_step": int(total_samples) * raster_elem_size(args.workload)}
                           if dec_e2e_ms else None),
                   "kernels_ms": mean_ms(dec_prof),
                   "roofline": roof(dec_prof.get("k_decode_subframes"), dec_alg, "k_decode_subframes",
                                    ("compressed bytes read + raster pixels written by the fused skim + Rice decode + predictor restore + "
                                     "denormalise launch" if fused_dec else "compressed bytes read + int32 audio written") +
                                    "; issue-bound (ALU pipe), not HBM-bound: `issue` holds the fraction of the integer issue roofline",
                                    MODEL_OPS["decode"])},
        "kernels_ms": mean_ms(enc_prof),
        "roofline": roof(enc_prof.get("k_enc_code") or enc_prof.get("subframe_analysis_total"), enc_alg, "k_enc_code",
                         "planar audio read + compressed bytes written by the dominant encode kernel (residual, Rice search, bit packing); "
                         "issue-bound, not HBM-bound (see DESIGN.md)", MODEL_OPS["encode_l8" if level >= 6 else "encode_l5"]),
        "cpu_baseline": cpu,
        "e2e": {"value": total_samples / (e2e_ms * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": int(total_samples) * raster_elem_size(args.workload), "d2h_bytes_per_step": nout_total},
        "weak": ({"value": samples_scene * world / (weak_ms * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": weak_ms,
                  "note": "every rank codes a whole scene (round 1's number); secondary"} if weak_ms else None),
        "container_check": container,
        "c5_bbox": c5_line(c5, c5_ms, world),
        "gpu_launches": int(tot[1]),
        "clocks": clocks,
    }
    emit_line(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def raster_elem_size(workload: str) -> int:
    return 4 if workload == "c4" else 2


# --dump-outputs: outputs larger than DUMP_SAMPLE elements (the frame bytes, the decoded raster) are kept as a sample at
# positions drawn from a fixed seed, so that two builds can be compared output for output within DUMP_LIMIT bytes
DUMP_SAMPLE = 1 << 22
DUMP_LIMIT = 64 << 20


def sample_positions(n_total: int, seed: int) -> np.ndarray:
    if n_total <= DUMP_SAMPLE:
        return np.arange(n_total, dtype=np.int64)
    return np.sort(np.random.default_rng(seed).integers(0, n_total, DUMP_SAMPLE, dtype=np.int64))


def encode_outputs(enc) -> dict:
    """What Engine.encode_tiles returned (EncodedTiles): integers as float64 (exact), frame bytes sampled as float32."""
    import torch
    pos = torch.from_numpy(sample_positions(int(enc.payload.numel()), seed=1)).to(enc.payload.device)
    res = {"encode_payload_sample": enc.payload[pos].cpu().numpy().astype(np.float32)}
    for name in ("offsets", "sizes", "minmax", "n_samples", "sample_rates"):
        res["encode_" + name] = np.asarray(getattr(enc, name), dtype=np.float64)
    for name in ("frame_bytes", "sub_bitoff"):             # int32 views of uint32 data
        res["encode_" + name] = getattr(enc, name).cpu().numpy().view(np.uint32).astype(np.float64)
    return res


def decode_outputs(out, status) -> dict:
    """What Engine.decode_tiles produced: the raster it wrote (sampled; uint16, int16 and float32 are exact in float32) and
    the status words it returned."""
    import torch
    flat = (out.view(torch.int16) if out.dtype == torch.uint16 else out).reshape(-1)
    vals = flat[torch.from_numpy(sample_positions(flat.numel(), seed=2)).to(flat.device)].cpu().numpy()
    if out.dtype == torch.uint16:
        vals = vals.view(np.uint16)
    return {"decode_raster_sample": vals.astype(np.float32), "decode_status": np.asarray(status, dtype=np.float64)}


def write_outputs(directory: str, arrays: dict) -> None:
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT, f"--dump-outputs: {total} bytes exceed {DUMP_LIMIT}"
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)
    print(f"[bench] wrote {len(arrays)} arrays ({total} bytes) to {directory}", file=sys.stderr)


def _scratch_dir(rank, world, dev):
    """A directory every rank of this node sees (rank 0 creates it, the name is broadcast)."""
    import torch
    import torch.distributed as dist
    base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
    name = [tempfile.mkdtemp(prefix="frb_bench_", dir=base) if rank == 0 else None]
    if world > 1:
        dist.broadcast_object_list(name, src=0)
    return name[0]


def container_check(args, eng, rank, world, dev, host_raster, r0, full_shape, ts, level, tiles_all):
    """All ranks write ONE streaming container (distributed.encode_streaming_sharded from their host slabs); rank 0 opens it
    with the public SpatialFLACStreamer, decodes the first tile of three different ranks and compares them with the source."""
    import torch
    import torch.distributed as dist
    from flac_raster_b200.distributed import encode_streaming_sharded, tile_shards
    from flac_raster_b200.spatial_encoder import SpatialFLACStreamer

    d = _scratch_dir(rank, world, dev)
    path = os.path.join(d, "scene.flac")
    transform = (10.0, 0.0, 399960.0, 0.0, -10.0, 4500000.0)           # a UTM-like north-up grid
    dtype_name = "uint16" if args.workload == "c3" else "int16"
    t0 = time.perf_counter()
    index, enc, (a, b) = encode_streaming_sharded(host_raster, r0, full_shape, transform, "EPSG:32633", None, dtype_name, ts, level,
                                                  path, rank, world, engine=eng)
    wall = time.perf_counter() - t0
    res = None
    if rank == 0:
        size = os.path.getsize(path)
        s = SpatialFLACStreamer(path)
        want_size = s.header_size + sum(f["byte_size"] for f in index["frames"])
        picks = sorted({tile_shards(tiles_all, world)[r][0] for r in (0, world // 2, world - 1)} | {len(tiles_all) - 1})
        ok = size == want_size and len(s.spatial_index.frames) == len(tiles_all)
        for tid in picks:
            tile, meta = s.get_tile_by_id(tid)
            t = tiles_all[tid]
            src = make_rows(args.workload, dev, int(t["row_off"]), int(t["row_off"] + t["h"]), args.scale_div)
            src = src[:, :, int(t["col_off"]):int(t["col_off"] + t["w"])]
            src_np = src.view(torch.int16).cpu().numpy().view(tile.dtype) if src.dtype == torch.uint16 else src.cpu().numpy()
            ok = ok and tile.shape == src_np.shape and bool(np.array_equal(tile, src_np))
        res = {"ok": bool(ok), "bytes": size, "tiles_verified": picks, "write_wall_s": wall,
               "path": "distributed.encode_streaming_sharded -> write_sharded_container -> SpatialFLACStreamer.get_tile_by_id"}
        if world == 1 and ok:
            # the whole scene back through the public call (file in page cache -> pinned staging -> H2D -> fused decode -> D2H ->
            # one array per tile): the read direction of the same container, wall clock of the second call
            bb = (-1e12, -1e12, 1e12, 1e12)
            got = s.get_tiles_by_bbox(*bb)
            del got
            t1 = time.perf_counter()
            got = s.get_tiles_by_bbox(*bb)
            dt = time.perf_counter() - t1
            n_px = sum(int(a.size) for a, _ in got)
            a_last, m_last = got[-1]
            t = tiles_all[-1]
            src = make_rows(args.workload, dev, int(t["row_off"]), int(t["row_off"] + t["h"]), args.scale_div)[:, :, int(t["col_off"]):int(t["col_off"] + t["w"])]
            src_np = src.view(torch.int16).cpu().numpy().view(a_last.dtype) if src.dtype == torch.uint16 else src.cpu().numpy()
            res["bbox_all"] = {"ok": bool(len(got) == len(tiles_all) and np.array_equal(a_last, src_np)), "ms_per_call": 1e3 * dt,
                               "value": n_px / dt / 1e9, "unit": UNIT, "tiles": len(got)}
            res["ok"] = bool(res["ok"] and res["bbox_all"]["ok"])
            del got
    if world > 1:
        dist.barrier()
    if rank == 0:
        shutil.rmtree(d, ignore_errors=True)
    return res


def c5_bbox_sweep(eng, rank, world, dev, barrier, reps: int = 3):
    """BASELINE.json configs[4]: get_tiles_by_bbox over 4096 tiles of 512x512 int16 through the public API; each rank fetches
    and decodes its share of the requested tiles (no collective) from a container in /dev/shm (page cache)."""
    import torch
    import torch.distributed as dist
    from flac_raster_b200 import synth
    from flac_raster_b200.distributed import encode_streaming_sharded, shard_plan
    from flac_raster_b200.spatial_encoder import SpatialFLACStreamer

    n_tiles, T = 4096, 512
    H, W = n_tiles * T, T
    d = _scratch_dir(rank, world, dev)
    path = os.path.join(d, "c5.flac")
    tiles_all, (a, b), (r0, r1) = shard_plan(H, W, T, rank, world)
    slab = synth.dem_int16_tiles(b - a, T, device=dev, first_tile=a)
    transform = (1.0, 0.0, 0.0, 0.0, -1.0, float(H))
    encode_streaming_sharded(slab, r0, (1, H, W), transform, "EPSG:32633", None, "int16", T, 5, path, rank, world, engine=eng)
    barrier()
    s = SpatialFLACStreamer(path)
    res = s.get_tiles_by_bbox(-1.0, -1.0, W + 1.0, H + 1.0)                 # warm-up (buffers, page cache)
    assert len(res) == b - a, (len(res), a, b)
    ok = True
    for k in (0, len(res) // 2, len(res) - 1):
        tile, meta = res[k]
        ok = ok and meta["frame_id"] == a + k and bool(np.array_equal(tile, slab[:, k * T:(k + 1) * T].cpu().numpy()))
    del res
    times = []
    for _ in range(reps):
        barrier()
        t0 = time.perf_counter()
        res = s.get_tiles_by_bbox(-1.0, -1.0, W + 1.0, H + 1.0)
        times.append((time.perf_counter() - t0) * 1e3)
        n_got = len(res)
        del res
    barrier()
    size = os.path.getsize(path) if rank == 0 else 0
    if world > 1:
        dist.barrier()
    if rank == 0:
        shutil.rmtree(d, ignore_errors=True)
    return {"ms": float(np.median(times)), "ok": bool(ok), "tiles_this_rank": n_got, "bytes": size, "ms_all": times}


def c5_line(c5, ms_max, world):
    if not c5:
        return None
    if "error" in c5:
        return c5
    samples = 4096 * 512 * 512
    return {"value": samples / (ms_max * 1e-3) / 1e9, "unit": UNIT, "ms_per_call": ms_max, "ok": c5["ok"], "container_bytes": c5["bytes"],
            "n_gpus": world, "tiles": 4096, "tiles_rank0": c5["tiles_this_rank"],
            "what": "SpatialFLACStreamer.get_tiles_by_bbox over all 4096 tiles of 512x512 int16 (BASELINE.json configs[4]), wall clock of the "
                    "public call on the slowest rank: file ranges (page cache) -> pinned staging -> H2D -> fused decode -> D2H -> one array per tile; "
                    "requested tiles split over the ranks, no collective"}


if __name__ == "__main__":
    sys.exit(main())
