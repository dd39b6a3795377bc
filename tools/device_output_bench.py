#!/usr/bin/env python3
"""Frames delivered to device memory against the packed host read-back, on bench.py's end-to-end workload (512
synthetic 1080p streams x 30 frames, bitstream parsed on the device, 4 time steps in flight).

Arms, alternated over --rounds rounds:
  packed_i420 : PackKernel into engine staging + one D2H copy per time step into a pinned ring (what bench.py times)
  device_i420 : PackKernel straight into a CUDA tensor ring (vp8r_read_batch_device, VP8R_LAYOUT_I420)
  device_rgb  : ConvertRgbKernel into a CUDA tensor ring (VP8R_LAYOUT_RGB24)
For each: end-to-end frames/s (bench.py's loop: one set of streams after another, the last pass drains), the read-back
alone (CUDA events around --reps calls on one decoded batch, ms per batch of all streams), its algorithmic bytes
(read + written: 3 B/pixel for I420, 4.5 B/pixel for RGB24) per second and their share of bench.peak_hbm().  The
outputs of the timed calls of a sample of streams are compared with the host read-back (and, for RGB, with the integer
BT.601 conversion in numpy); any difference fails the run.  One JSON document goes to --out.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

import bench  # noqa: E402

W, H, FB = bench.W, bench.H, bench.FRAME_BYTES
ARMS = ["packed_i420", "device_i420", "device_rgb"]


def rgb_from_i420(img):
    a = np.frombuffer(img, np.uint8)
    cw, ch = W // 2, H // 2
    y = a[:W * H].reshape(H, W).astype(np.int32) - 16
    u = a[W * H:W * H + cw * ch].reshape(ch, cw).repeat(2, 0).repeat(2, 1).astype(np.int32) - 128
    v = a[W * H + cw * ch:].reshape(ch, cw).repeat(2, 0).repeat(2, 1).astype(np.int32) - 128
    rgb = np.stack([(298 * y + 409 * v + 128) >> 8, (298 * y - 100 * u - 208 * v + 128) >> 8, (298 * y + 516 * u + 128) >> 8], -1)
    return np.clip(rgb, 0, 255).astype(np.uint8)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else f"nvidia-smi failed: {q.stderr.strip()}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=512)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--passes", type=int, default=3, help="end-to-end passes per arm and round (bench.py --e2e-steps)")
    ap.add_argument("--reps", type=int, default=50, help="read-back calls timed on one decoded batch")
    ap.add_argument("--sample", type=int, default=8, help="streams whose outputs are compared")
    ap.add_argument("--out", required=True)
    args = ap.parse_args()

    import torch
    import vp8_b200
    if not torch.cuda.is_available():
        raise SystemExit("device_output_bench.py needs a GPU")
    S, depth = args.streams, 4
    stream = torch.cuda.Stream()
    eng = vp8_b200.Engine(0, cuda_stream=stream.cuda_stream)
    tmp = tempfile.mkdtemp()
    paths = [os.path.join(tmp, f"s{k}.ivf") for k in range(S)]
    with ThreadPoolExecutor(max_workers=os.cpu_count()) as ex:
        list(ex.map(lambda k: bench.synth_stream(7122 + k, paths[k]), range(S)))
    payloads = [vp8_b200.read_ivf(p)[1] for p in paths]
    shutil.rmtree(tmp, ignore_errors=True)

    pinned = [torch.empty((S, FB), dtype=torch.uint8, pin_memory=True) for _ in range(depth)]
    rings = {"device_i420": ([torch.empty((S, FB), dtype=torch.uint8, device="cuda") for _ in range(depth)], "i420"),
             "device_rgb": ([torch.empty((S, H, W, 3), dtype=torch.uint8, device="cuda") for _ in range(depth)], "rgb")}
    decs = {a: vp8_b200.BatchDecoder(eng, S, parse_threads=os.cpu_count(), pinned=True, device_parse=True, depth=depth)
            for a in ARMS}
    host = torch.empty((args.sample, FB), dtype=torch.uint8, pin_memory=True)
    sample = list(range(0, S, max(1, S // args.sample)))[:args.sample]

    def outputs(arm):
        return {"out_packed": (tuple(r.data_ptr() for r in pinned), FB)} if arm == "packed_i420" else {"out_device": rings[arm]}

    def check(arm, dec, rows_of, what, only=None):
        """rows_of(i) = the arm's output for sample stream i (bytes); compared with the host read-back of that stream.
        only: the sample streams that have an output (the last step's shown frames)."""
        eng.read_batch_packed([dec.streams[i] for i in sample], host.data_ptr(), FB)
        for j, i in enumerate(sample):
            if only is not None and i not in only:
                continue
            want = host[j].numpy().tobytes()
            if arm == "device_rgb":
                want = rgb_from_i420(want).tobytes()
            if rows_of(i) != want:
                raise SystemExit(f"{arm}: {what}: stream {i} differs from the reference")

    result = {"gpu": gpu_info(), "workload": f"{S} synthetic 1080p streams x {bench.FRAMES} frames ({bench.SYNTH_ARGS}), "
              f"device parse, depth {depth}", "peak_hbm": dict(zip(("gb_per_s", "kind"), bench.peak_hbm())), "arms": {a: [] for a in ARMS}}
    for a in ARMS:  # warm-up: allocations, pinned buffers, module loads
        decs[a].decode(payloads, **outputs(a))
    torch.cuda.synchronize()
    for rnd in range(args.rounds):
        for arm in ARMS:
            dec = decs[arm]
            last = {}

            def on_step(t, live, frames, last=last):
                if t == bench.FRAMES - 1:
                    last["shown"] = [i for i, f in zip(live, frames) if f.desc().hdr.show_frame]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for k in range(args.passes):
                dec.reset()
                final = k + 1 == args.passes
                g_last = dec._g + bench.FRAMES - 1  # ring entry of this pass's last step
                dec.decode(payloads, drain=final, on_step=on_step if final else None, **outputs(arm))
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            fps = S * bench.FRAMES * args.passes / dt
            # the timed outputs: the last step of the last pass
            row = {i: k for k, i in enumerate(last["shown"])}
            if arm == "packed_i420":
                entry = pinned[g_last % depth]
                check(arm, dec, lambda i: entry[row[i]].numpy().tobytes(), "end-to-end output", row)
            else:
                entry = rings[arm][0][g_last % depth].cpu()
                check(arm, dec, lambda i: entry[row[i]].numpy().tobytes(), "end-to-end output", row)
            # the read-back alone, on the engine's stream
            n = S
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(stream):
                if arm == "packed_i420":
                    dst = pinned[0]
                    eng.read_batch_packed(dec.streams, dst.data_ptr(), FB, async_=True)
                    eng.sync()
                    t1 = time.perf_counter()
                    for _ in range(args.reps):
                        eng.read_batch_packed(dec.streams, dst.data_ptr(), FB, async_=True)
                    eng.sync()  # the D2H copies run on the engine's copy stream: host clock around a full drain
                    ms = (time.perf_counter() - t1) * 1e3 / args.reps
                    check(arm, dec, lambda i: dst[i].numpy().tobytes(), "read-back alone")
                else:
                    ring, layout = rings[arm]
                    eng.read_batch_device(dec.streams, ring[0], layout)
                    ev0.record(stream)
                    for _ in range(args.reps):
                        eng.read_batch_device(dec.streams, ring[0], layout)
                    ev1.record(stream)
                    ev1.synchronize()
                    ms = ev0.elapsed_time(ev1) / args.reps
                    out = ring[0].cpu()
                    check(arm, dec, lambda i: out[i].numpy().tobytes(), "read-back alone")
            alg = n * W * H * (4.5 if arm == "device_rgb" else 3.0)
            gbs = alg / (ms / 1e3) / 1e9
            rec = {"round": rnd, "e2e_frames_per_s": round(fps, 1), "e2e_seconds": round(dt, 3),
                   "readback_ms_per_batch": round(ms, 4), "batch_frames": n, "alg_bytes_per_batch": int(alg),
                   "alg_gb_per_s": round(gbs, 1), "frac_of_peak_hbm": round(gbs / result["peak_hbm"]["gb_per_s"], 4),
                   "readback_timing": "host clock around calls + sync (includes the D2H copy)" if arm == "packed_i420"
                   else "CUDA events on the engine stream"}
            result["arms"][arm].append(rec)
            print(arm, json.dumps(rec), flush=True)
    result["outputs_checked"] = f"streams {sample}: the last step of each timed end-to-end run and the read-back-alone output"
    for d in decs.values():
        d.close()
    eng.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({a: [r["e2e_frames_per_s"] for r in v] for a, v in result["arms"].items()}))


if __name__ == "__main__":
    main()
