#!/usr/bin/env python3
"""Inter-frame encoder throughput, split and compression on a B200.

Workload: --streams streams (default 64) of --width x --height (default 1920x1080), one key frame and --inter
inter frames each (default 29) of a seeded moving scene: per stream a smoothed random texture under its own
whole-pixel pan, plus a rectangle that moves across it and per-frame noise (the pictures are cut from one shared
texture, so building them costs little host time).  Every time step encodes all streams in one
vp8r_encode_inter_frames call (Engine.encode_inter_frames).

Reports, in one JSON document (--out):
  - inter frames/s: host clock around each synchronous inter call, summed over the timed steps (after --warmup steps);
  - the split of one inter call into kernels and the rest (host padding, staging copies, read-back, mode assignment):
    kernel times from torch.profiler with CUDA activities, in a separate run of --profile-steps calls;
  - bytes per inter frame against bytes per key frame of the same pictures at the same quantiser (the key frames of
    --compare-streams streams, encoded as key frames on streams of their own);
  - PSNR (Y, whole frame) of the reconstructions of --compare-streams streams against their source;
  - the card's name and power limit (nvidia-smi).
--input selects where the pictures come from: "host" (cropped I420 bytes, the default), "i420" (a CUDA tensor of the
same bytes) or "rgb" (a CUDA tensor of RGB24 pictures, made from the I420 pictures in numpy by include/vp8r.h's
YUV -> RGB formula).  A device input is uploaded before each call, outside the timed window; with "rgb" the PSNR is
measured against the I420 the encoder codes (Engine.convert_to_i420).
--intra-mbs lets the inter frames code macroblocks intra (Engine.encode_inter_frames(intra_mbs=True), B_PRED among the
candidates); the time of that pass per call is read from the engine's intra timer during the profiled calls.
--cut-every N replaces the picture of every stream with an unrelated scene (the texture turned by 180 degrees, and back)
every N frames.
--dry-run builds the pictures of the first two time steps and prints the plan without touching a device.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


class Scene:
    """Seeded moving scene of n streams: picture(s, t) is cropped I420 bytes."""

    def __init__(self, n, w, h, steps, seed=2024, cut_every=0):
        rng = np.random.default_rng(seed)
        self.w, self.h, self.n = w, h, n
        self.margin = 2 * steps + 40
        th, tw = h + 2 * self.margin, w + 2 * self.margin
        t = rng.integers(0, 256, (th + 2, tw + 2)).astype(np.float32)
        t = (t[:-2, :-2] + t[1:-1, :-2] + t[2:, :-2] + t[:-2, 1:-1] + 2 * t[1:-1, 1:-1] + t[2:, 1:-1] + t[:-2, 2:] + t[1:-1, 2:] + t[2:, 2:]) / 10
        self.tex = np.clip((t - 128) * 2.0 + 128, 0, 255).astype(np.uint8)
        self.tex_cut = np.ascontiguousarray(self.tex[::-1, ::-1])
        self.cut_every = cut_every
        self.vel = [(int(rng.integers(-2, 3)), int(rng.integers(-2, 3))) for _ in range(n)]
        self.off = [(int(rng.integers(0, 20)), int(rng.integers(0, 20))) for _ in range(n)]
        self.noise = [rng.integers(-2, 3, (h, w)).astype(np.int16) for _ in range(4)]
        cw, ch = (w + 1) // 2, (h + 1) // 2
        cy, cx = np.mgrid[0:ch, 0:cw]
        self.u = np.clip(118 + 30 * np.sin(cx / 23.0), 0, 255).astype(np.uint8).tobytes()
        self.v = np.clip(136 + 30 * np.cos(cy / 17.0), 0, 255).astype(np.uint8).tobytes()

    def picture(self, s, t):
        (vy, vx), (oy, ox) = self.vel[s], self.off[s]
        y0, x0 = self.margin + oy + vy * t - 20, self.margin + ox + vx * t - 20
        tex = self.tex_cut if self.cut_every and (t // self.cut_every) % 2 else self.tex
        y = tex[y0:y0 + self.h, x0:x0 + self.w].astype(np.int16) + self.noise[(s + t) % 4]
        rh, rw = self.h // 6, self.w // 6
        ry, rx = (self.h // 3 + 5 * t) % (self.h - rh), (self.w // 4 + 7 * t + 31 * s) % (self.w - rw)
        y[ry:ry + rh, rx:rx + rw] = 60 + 40 * ((np.arange(rw) // 6) % 2)
        return np.clip(y, 0, 255).astype(np.uint8).tobytes() + self.u + self.v


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else f"nvidia-smi failed: {q.stderr.strip()}"


def rgb_from_i420(img, w, h):
    """Cropped I420 bytes -> (h, w, 3) RGB by include/vp8r.h's BT.601 formula (chroma point-sampled)."""
    a = np.frombuffer(img, np.uint8)
    cw, ch = (w + 1) // 2, (h + 1) // 2
    y = a[:w * h].reshape(h, w).astype(np.int32) - 16
    u = a[w * h:w * h + cw * ch].reshape(ch, cw).repeat(2, 0).repeat(2, 1)[:h, :w].astype(np.int32) - 128
    v = a[w * h + cw * ch:].reshape(ch, cw).repeat(2, 0).repeat(2, 1)[:h, :w].astype(np.int32) - 128
    rgb = np.stack([(298 * y + 409 * v + 128) >> 8, (298 * y - 100 * u - 208 * v + 128) >> 8, (298 * y + 516 * u + 128) >> 8], -1)
    return np.clip(rgb, 0, 255).astype(np.uint8)


def psnr_y(a, b, n):
    a = np.frombuffer(a, np.uint8)[:n].astype(np.float64)
    b = np.frombuffer(b, np.uint8)[:n].astype(np.float64)
    mse = float(np.mean((a - b) ** 2))
    return 99.0 if mse == 0 else 10 * np.log10(255.0 ** 2 / mse)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--streams", type=int, default=64)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--inter", type=int, default=29, help="inter frames per stream after its key frame")
    ap.add_argument("--warmup", type=int, default=2, help="inter steps not timed")
    ap.add_argument("--q", type=int, default=40)
    ap.add_argument("--lf", type=int, default=16)
    ap.add_argument("--search-range", type=int, default=16)
    ap.add_argument("--compare-streams", type=int, default=4, help="streams whose key-frame sizes and PSNR are measured")
    ap.add_argument("--profile-steps", type=int, default=3)
    ap.add_argument("--input", choices=("host", "i420", "rgb"), default="host", help="where the pictures come from")
    ap.add_argument("--intra-mbs", action="store_true", help="intra macroblocks in inter frames")
    ap.add_argument("--cut-every", type=int, default=0, help="an unrelated scene every N frames (0: never)")
    ap.add_argument("--out", default=None)
    ap.add_argument("--dry-run", action="store_true", help="build the pictures of two steps and print the plan; no device")
    args = ap.parse_args()
    if args.warmup >= args.inter:
        raise SystemExit("--warmup must be smaller than --inter")
    n, w, h = args.streams, args.width, args.height
    scene = Scene(n, w, h, args.inter + 1, cut_every=args.cut_every)
    ncmp = min(args.compare_streams, n)
    plan = {"streams": n, "width": w, "height": h, "inter_frames_per_stream": args.inter, "timed_steps": args.inter - args.warmup,
            "q_index": args.q, "loop_filter_level": args.lf, "search_range": args.search_range, "compare_streams": ncmp,
            "input": args.input, "intra_mbs": args.intra_mbs, "cut_every": args.cut_every}
    if args.dry_run:
        t0 = time.perf_counter()
        pics = [scene.picture(s, t) for t in range(2) for s in range(n)]
        fb = w * h + 2 * ((w + 1) // 2) * ((h + 1) // 2)
        assert all(len(p) == fb for p in pics)
        plan["host_picture_build_s_per_step"] = (time.perf_counter() - t0) / 2
        print(json.dumps({"dry_run": plan}, indent=1))
        return 0

    import torch
    import vp8_b200
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: the encoder benchmark runs on the GPU only")
    eng = vp8_b200.Engine(0)

    def source(pics):
        """The encoder's input for one step and the I420 pictures it codes (bytes)."""
        if args.input == "host":
            return pics, pics, "i420"
        if args.input == "i420":
            dev = torch.from_numpy(np.frombuffer(b"".join(pics), np.uint8).reshape(n, -1)).cuda()
            torch.cuda.synchronize()
            return dev, pics, "i420"
        dev = torch.from_numpy(np.stack([rgb_from_i420(p, w, h) for p in pics])).cuda()
        coded = [bytes(r) for r in eng.convert_to_i420(dev, "rgb", w, h).cpu().numpy()]
        torch.cuda.synchronize()
        return dev, coded, "rgb"

    streams = [eng.open_stream() for _ in range(n)]
    key_streams = [eng.open_stream() for _ in range(ncmp)]
    fb_y = w * h
    step_s, inter_bytes, key_bytes, psnr = [], [], [], []
    intra_mbs = all_mbs = 0
    try:
        src, _, layout = source([scene.picture(s, 0) for s in range(n)])
        for f in eng.encode_key_frames(streams, src, w, h, args.q, args.lf, layout=layout):
            f.close()
        for t in range(1, args.inter + 1):
            src, pics, layout = source([scene.picture(s, t) for s in range(n)])
            t0 = time.perf_counter()
            frames = eng.encode_inter_frames(streams, src, w, h, args.q, args.lf, search_range=args.search_range, layout=layout,
                                             intra_mbs=args.intra_mbs)
            dt = time.perf_counter() - t0
            if t > args.warmup:
                step_s.append(dt)
            for f in frames:
                d = f.desc().hdr
                intra_mbs += d.mb_cols * d.mb_rows - d.n_inter_mbs
                all_mbs += d.mb_cols * d.mb_rows
            for s in range(ncmp):
                inter_bytes.append(len(frames[s].write_bitstream()))
                psnr.append(psnr_y(streams[s].read_frame(), pics[s], fb_y))
            for f in frames:
                f.close()
            # the same pictures as key frames, for the size comparison
            kf = eng.encode_key_frames(key_streams, pics[:ncmp], w, h, args.q, args.lf)
            key_bytes += [len(f.write_bitstream()) for f in kf]
            for f in kf:
                f.close()
        # separate run under the profiler: kernel times of --profile-steps inter calls
        from torch.profiler import ProfilerActivity, profile
        src, _, layout = source([scene.picture(s, args.inter + 1) for s in range(n)])
        eng.set_timing(True)
        eng.timers(reset=True)
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            t0 = time.perf_counter()
            for _ in range(args.profile_steps):
                for f in eng.encode_inter_frames(streams, src, w, h, args.q, args.lf, search_range=args.search_range,
                                                 layout=layout, intra_mbs=args.intra_mbs):
                    f.close()
            prof_wall = time.perf_counter() - t0
        tm = eng.timers()
        eng.set_timing(False)
        kernels, copies = {}, {}
        for ev in prof.key_averages():
            dev_us = getattr(ev, "self_device_time_total", None)
            if dev_us is None:
                dev_us = getattr(ev, "self_cuda_time_total", 0)
            if not dev_us or ev.key.startswith("cuda"):
                continue
            (copies if ev.key.startswith(("Memcpy", "Memset")) else kernels)[ev.key] = dev_us / 1e3 / args.profile_steps
        kernel_ms = sum(kernels.values())
    finally:
        for st in streams + key_streams:
            st.close()
        eng.close()
    total = sum(step_s)
    res = {
        "workload": plan,
        "gpu": gpu_info(),
        "inter_frames_per_s": n * len(step_s) / total,
        "inter_call_ms": {"mean": 1e3 * total / len(step_s), "min": 1e3 * min(step_s), "max": 1e3 * max(step_s)},
        "profile": {"calls": args.profile_steps, "wall_ms_per_call_under_profiler": 1e3 * prof_wall / args.profile_steps,
                    "kernel_ms_per_call": kernels, "kernels_total_ms_per_call": kernel_ms, "copy_ms_per_call": copies,
                    "rest_ms_per_call": 1e3 * prof_wall / args.profile_steps - kernel_ms,
                    "note": "rest = host padding and staging copies (host input), read-back copies, mode assignment (wall under the "
                            "profiler minus kernel time)"},
        "intra_timer_ms_per_call": tm.ms_intra / args.profile_steps,
        "intra_mb_fraction": intra_mbs / max(all_mbs, 1),
        "bytes_per_inter_frame": float(np.mean(inter_bytes)),
        "bytes_per_key_frame_same_pictures": float(np.mean(key_bytes)),
        "inter_over_key": float(np.mean(inter_bytes) / np.mean(key_bytes)),
        "psnr_y_inter_db": {"mean": float(np.mean(psnr)), "min": float(np.min(psnr))},
    }
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
