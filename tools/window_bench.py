"""Windowed reads of C3 (10980 x 10980 uint16 x 8 bands, synthetic Sentinel-2-like) against a full decode plus crop.

Two layouts of the same scene: one FLAC file (29 434 frames of 4096 samples) and a tile-1024 streaming container.  For
windows of 256^2, 1024^2 and 4096^2 pixels at seeded positions it times
  * device-resident: frames already in HBM -> the window in HBM (Engine.decode_window, against Engine.decode_tiles of the
    whole scene plus a crop), host synchronisation included;
  * end to end from a page-cached file: RasterFLACConverter.read_window / SpatialFLACStreamer.read_bbox, against
    flac_to_array / get_tiles_by_bbox stitched, each plus a crop.
Every window is checked against the full decode.  Prints one JSON line (medians in ms, frames decoded, GPU name and
power limit).  Files go to a temporary directory that is removed at the end.

    python tools/window_bench.py [--steps 5] [--warmup 1] [--seed 0]
"""
from __future__ import annotations

import argparse
import json
import shutil
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, limit = (v.strip() for v in out.split(","))
        return name, limit
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})", "unknown"


def timed(fn, steps, warmup):
    import torch
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(steps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--sizes", default="256,1024,4096")
    args = ap.parse_args()

    import torch
    from flac_raster_b200 import flacfmt, synth
    from flac_raster_b200.converter import RasterFLACConverter, build_flac_file, tile_metadata
    from flac_raster_b200.engine import Engine, tile_grid, window_frames
    from flac_raster_b200.spatial_encoder import SpatialFLACStreamer, build_streaming_container, write_streaming_container

    torch.cuda.set_device(0)
    eng = Engine(0)
    import flac_raster_b200.engine as engine_mod
    engine_mod._default_engine = eng
    bands, H, W = 8, 10980, 10980
    raster = synth.sentinel2_like(H, W, bands, device=eng.device)
    rng = np.random.default_rng(args.seed)
    sizes = [int(s) for s in args.sizes.split(",")]
    windows = []
    for s in sizes:
        c0, r0 = int(rng.integers(0, W - s + 1)), int(rng.integers(0, H - s + 1))
        windows.append((c0, r0, s, s))
    tmp = Path(tempfile.mkdtemp(prefix="frb_window_bench_"))
    result = {"workload": "c3 window reads", "windows": [list(w) for w in windows], "steps": args.steps}
    try:
        layouts = {}
        # ---- one file
        one_tiles = tile_grid(H, W, W)
        enc1 = eng.encode_tiles(raster, one_tiles, 5, payload_name="wb_payload1")
        fb1 = enc1.frame_bytes.cpu().numpy().view(np.uint32)
        sb1 = enc1.sub_bitoff.cpu().numpy().view(np.uint32)
        md = tile_metadata(W, H, bands, "uint16", None, None, float(enc1.minmax[0, 0]), float(enc1.minmax[0, 1]), None, 32767)
        path1 = tmp / "c3_one.flac"
        path1.write_bytes(build_flac_file(enc1.payload.cpu().numpy().tobytes(), H * W, bands, enc1.bps, int(enc1.sample_rates[0]),
                                          enc1.blocksize, md, padding=1024,
                                          seek_index=flacfmt.pack_seek_index(bands, enc1.blocksize, fb1, sb1)))
        payload1 = eng._buf("wb_data1", enc1.payload.numel() + 64)
        payload1[:enc1.payload.numel()].copy_(enc1.payload)
        layouts["one_file"] = (one_tiles, enc1, payload1, (fb1, sb1))
        del enc1
        # ---- tile-1024 container
        idx, headers, enc2 = build_streaming_container(raster, (1.0, 0.0, 0.0, 0.0, -1.0, 0.0), "", None, "uint16", 1024)
        path2 = tmp / "c3_t1024.flac"
        write_streaming_container(path2, idx, headers, enc2.payload.cpu().numpy(), enc2.offsets, enc2.sizes)
        payload2 = eng._buf("wb_data2", enc2.payload.numel() + 64)
        payload2[:enc2.payload.numel()].copy_(enc2.payload)
        layouts["tile1024"] = (tile_grid(H, W, 1024), enc2, payload2,
                               (enc2.frame_bytes.cpu().numpy().view(np.uint32), enc2.sub_bitoff.cpu().numpy().view(np.uint32)))
        result["file_bytes"] = {"one_file": path1.stat().st_size, "tile1024": path2.stat().st_size}
        del raster
        torch.cuda.empty_cache()

        full = torch.empty((bands, H, W), dtype=torch.uint16, device=eng.device)
        dev = {}
        for name, (tiles, enc, data, index) in layouts.items():
            def full_decode():
                st = eng.decode_tiles(data, enc.offsets, enc.sizes, tiles, enc.sample_rates, enc.minmax, 32767.0, full, 16,
                                      enc.blocksize, index=index)
                assert not (st[0] or st[1] or st[2])
            row = {"full_decode_ms": timed(full_decode, args.steps, args.warmup)}
            full_decode()
            for (c0, r0, w, h) in windows:
                out = torch.empty((bands, h, w), dtype=torch.uint16, device=eng.device)
                status = {}

                def win_decode():
                    status["s"] = eng.decode_window(data, enc.offsets, enc.sizes, tiles, enc.sample_rates, enc.minmax, 32767.0,
                                                    (c0, r0, w, h), out, 16, enc.blocksize, index=index)

                def full_crop():
                    full_decode()
                    return full[:, r0:r0 + h, c0:c0 + w].clone()

                ms = timed(win_decode, args.steps, args.warmup)
                ms_full = timed(full_crop, args.steps, args.warmup)
                match = bool(torch.equal(out, full_crop()))
                runs = window_frames(tiles, (c0, r0, w, h), enc.blocksize)
                row[f"{w}x{h}"] = {"window_ms": ms, "full_plus_crop_ms": ms_full, "frames_decoded": int(status["s"][3]),
                                   "frames_total": int(enc.frames_per_tile().sum()), "runs": len(runs), "equal": match}
            dev[name] = row
        result["device_resident"] = dev
        del full, layouts
        torch.cuda.empty_cache()

        conv = RasterFLACConverter()
        streamer = SpatialFLACStreamer(path2)
        full1, _ = conv.flac_to_array(path1)
        e2e = {"one_file": {}, "tile1024": {}}
        e2e["one_file"]["full_decode_ms"] = timed(lambda: conv.flac_to_array(path1), max(1, args.steps // 2), 1)
        for (c0, r0, w, h) in windows:
            want = full1[:, r0:r0 + h, c0:c0 + w]
            got = {}

            def one():
                got["a"], got["m"] = conv.read_window(path1, c0, r0, w, h)

            def one_full():
                a, _ = conv.flac_to_array(path1)
                return a[:, r0:r0 + h, c0:c0 + w].copy()

            bbox = (c0 + 0.5, -(r0 + h) + 0.5, c0 + w - 0.5, -r0 - 0.5)

            def cont():
                got["b"], got["n"] = streamer.read_bbox(*bbox)

            def cont_full():
                canvas = np.empty((bands, H, W), dtype=np.uint16)
                for arr, m in streamer.get_tiles_by_bbox(*bbox, shard=False):
                    wn = m["window"]
                    canvas[:, wn["row_off"]:wn["row_off"] + wn["height"], wn["col_off"]:wn["col_off"] + wn["width"]] = arr
                return canvas[:, r0:r0 + h, c0:c0 + w].copy()

            ms1 = timed(one, args.steps, args.warmup)
            ms2 = timed(cont, args.steps, args.warmup)
            e2e["one_file"][f"{w}x{h}"] = {"read_window_ms": ms1, "frames_decoded": got["m"]["frames_decoded"],
                                           "equal": bool(np.array_equal(got["a"], want))}
            e2e["tile1024"][f"{w}x{h}"] = {"read_bbox_ms": ms2, "stitched_tiles_plus_crop_ms": timed(cont_full, args.steps, args.warmup),
                                           "frames_decoded": got["n"]["frames_decoded"],
                                           "equal": bool(np.array_equal(got["b"], want)) and bool(np.array_equal(cont_full(), want))}
        result["end_to_end_page_cached"] = e2e
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    name, limit = gpu_info()
    result["gpu"] = name
    result["power_limit"] = limit
    print(json.dumps(result))


if __name__ == "__main__":
    main()
