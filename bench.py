#!/usr/bin/env python3
"""bench.py -- decoded 1080p frames/s of the VP8 reconstruction path on N B200s.

Workload (config.workload): S independent synthetic 1920x1080 streams per GPU, 30 frames each
(1 key + 29 inter, six-tap MC, normal loop filter on, segmentation, golden/altref updates, one
hidden alt-ref), written by tools/vp8synth.cc with seeds 7122+k.  A "step" decodes all S*30 frames
of a GPU once.  Streams are independent, so N GPUs = N*S streams, no collective (scaling: weak).

  value : decoded frames/s of the RECONSTRUCTION KERNELS with the parsed frames already resident in HBM
          (CUDA events on the launch stream, max over ranks); bitstream parse, H2D and read-back are not in
          it -- they are in e2e
  e2e   : decoded frames/s through the public API from compressed frames in host memory to cropped I420 of
          every SHOWN frame in pinned host memory: parse + H2D + kernels + D2H inside the timed region.
          This is the number to hold against the reference arm.
  roofline : algorithmic bytes (SURVEY 8(d): 1.5*Wa*Ha*(1+is_inter) + 32*coded blocks per frame)
          over the device time of ALL reconstruction kernels, against MEASURED_PEAKS.json hbm_gbs;
          roofline.per_kernel gives the same bytes attributed to the loop filter / motion compensation
          over that kernel's own device time (per launch = one batch of S frames); roofline.secondary is
          the ceiling that binds first on this path, instruction issue (warp instructions per frame from the
          committed ncu capture against 148 SMs x 4 issue slots x the SM clock)
  cpu_baseline : the reference decoder (oracle/_ref/decode[_native], compiled unmodified from the
          reference sources with -O3 -flto) on the host cores, one process per stream, on a bounded sample
  parity_checked : the first streams of the workload decoded through the public API and by that reference
          decoder: MD5 of every shown frame compared (exit code 1 on a mismatch)
  configs : BASELINE.json configs 3, 4 and 5 (one 1080p stream; 64 streams in total over the N GPUs;
          one 4K long-GOP stream cut at key frames into 8 segments over the N GPUs), kernel-only and end to end

--impl reference times that CPU decoder alone (the reference has no GPU path).
--dump-outputs DIR writes what the timed replay left in the streams after its last step (see dump_outputs), so
that two builds can be compared output for output: the inputs are the same from run to run for the same arguments.
"""
import argparse
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H, FRAMES = 1920, 1080, 30
FRAME_BYTES = W * H * 3 // 2
SYNTH = os.path.join(ROOT, "vp8_b200", "_lib", "vp8synth")
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
SYNTH_ARGS = "--width 1920 --height 1080 --frames 30 --log2-parts 2 --q 40 --lf 24 --pct-skip 55 --coef-density 3 --pct-empty-block 80"
# BASELINE config 5: one 3840x2160 stream, a key frame every 4 frames, 8 key-frame-delimited segments
UHD_ARGS = "--width 3840 --height 2160 --frames 32 --key-interval 4 --log2-parts 3 --q 40 --lf 24 --pct-skip 55 --coef-density 3 --pct-empty-block 80 --seed 9001"
UHD_FRAME_BYTES = 3840 * 2160 * 3 // 2


def synth_stream(seed, path, frames=FRAMES):
    args = SYNTH_ARGS.replace("--frames 30", f"--frames {frames}").split()
    subprocess.check_call([SYNTH] + args + ["--seed", str(seed), "--out", path])


def peak_hbm():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


_REF = None


def ref_decoder():
    """(path, description) of the reference decoder binary to time: the -march=native build when it runs on
    this host (BASELINE.md section 3), else the portable -march=x86-64-v3 one; (None, why) without either."""
    global _REF
    if _REF is not None:
        return _REF
    native, portable = os.path.join(REF_DIR, "decode_native"), os.path.join(REF_DIR, "decode")
    _REF = (None, "oracle/_ref/decode was not built")
    with tempfile.TemporaryDirectory() as td:
        probe = os.path.join(td, "p.ivf")
        try:
            subprocess.check_call([SYNTH, "--width", "64", "--height", "64", "--frames", "2", "--seed", "1", "--out", probe])
        except Exception:
            return _REF
        for path, what in ((native, None), (portable, "g++ -O3 -flto -march=x86-64-v3")):
            if not os.path.exists(path):
                continue
            try:
                ok = subprocess.run([path, probe, os.path.join(td, "o.yuv")], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL,
                                    timeout=60).returncode == 0
            except Exception:
                ok = False
            if ok:
                if what is None:
                    try:
                        what = open(native + ".flags").read().strip()
                    except Exception:
                        what = "g++ -O3 -flto -march=native"
                _REF = (path, what)
                break
    return _REF


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].startswith("Active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons}


def run_reference_cpu(paths, procs, keep_md5=False, frame_bytes=FRAME_BYTES):
    """Decodes `paths` with the reference decoder, `procs` processes at a time.  Returns (seconds, md5s) where
    md5s[k] = MD5 of every frame the decoder wrote for paths[k] (keep_md5; hashed after the clock stopped)."""
    binary = ref_decoder()[0]
    out_dir = tempfile.mkdtemp(dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    md5s = [None] * len(paths)
    t0 = time.perf_counter()
    running, todo = [], list(enumerate(paths))
    try:
        while todo or running:
            while todo and len(running) < procs:
                k, p = todo.pop(0)
                out = os.path.join(out_dir, f"o{k}.yuv" if keep_md5 else f"o{k % procs}.yuv")
                running.append((subprocess.Popen([binary, p, out]), k, out))
            proc, k, out = running[0]
            proc.wait()
            if proc.returncode != 0:
                raise RuntimeError("reference decoder failed")
            running.pop(0)
        dt = time.perf_counter() - t0
        if keep_md5:
            for k in range(len(paths)):
                with open(os.path.join(out_dir, f"o{k}.yuv"), "rb") as f:
                    md5s[k] = []
                    while True:
                        b = f.read(frame_bytes)
                        if not b:
                            break
                        md5s[k].append(hashlib.md5(b).hexdigest())
    finally:
        for r in running:
            r[0].kill()
        shutil.rmtree(out_dir, ignore_errors=True)
    return dt, md5s


def cpu_sample(cores, frames_per_stream, tmp):
    paths = []
    for k in range(cores):
        p = os.path.join(tmp, f"cpu{k}.ivf")
        synth_stream(7122 + k, p, frames_per_stream)
        paths.append(p)
    return paths


def reference_arm(args, rank, world):
    if rank != 0:
        return
    binary, flags = ref_decoder()
    if binary is None:
        print(json.dumps({"impl": "reference", "unavailable": flags}))
        return
    cores = os.cpu_count() or 1
    procs = min(cores, 64)
    with tempfile.TemporaryDirectory() as tmp:
        n_frames = 6  # per stream and step: ~1 s of CPU per process
        paths = cpu_sample(procs, n_frames, tmp)
        times = []
        for it in range(args.warmup + args.steps):
            dt, _ = run_reference_cpu(paths, procs)
            if it >= args.warmup:
                times.append(dt)
        total = sum(times)
        value = args.steps * procs * n_frames / total
    line = {
        "impl": "reference", "metric": "decoded 1080p frames/s", "value": value, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": f"reference CPU decoder ({os.path.basename(binary)}: {flags}), {procs} processes x one {n_frames}-frame "
                               "1080p synthetic stream per step (same generator settings and seeds as the GPU arm)",
                   "mp_per_s": value * W * H / 1e6},
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": procs, "kind": "reference",
                         "sample": f"{procs} streams x {n_frames} frames per step, one process per stream; {flags}"},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------
def kernel_only(torch, eng, stream, vp8_b200, payloads, passes, warm):
    """Parses + uploads `payloads` (list of streams, each a list of compressed frames) once and replays the
    reconstruction kernels.  Returns (milliseconds per pass, frames per pass, final checksums, decoder)."""
    S = len(payloads)
    steps = max(len(p) for p in payloads)
    dec = vp8_b200.BatchDecoder(eng, S, pinned=False)
    resident, frames_per_pass = [], 0
    for t in range(steps):
        live = [i for i in range(S) if len(payloads[i]) > t]
        frames = dec.parse_into([vp8_b200.ParsedFrame(pinned=False) for _ in live], [p[t] if len(p) > t else b"" for p in payloads], live)
        for f in frames:
            eng.upload(f, release_host=True)
        resident.append((live, frames))
        frames_per_pass += len(live)

    def one_pass():
        for live, frames in resident:
            eng.reconstruct_batch([dec.streams[i] for i in live], frames)

    for _ in range(warm):
        one_pass()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        ev0.record(stream)
        for _ in range(passes):
            one_pass()
        ev1.record(stream)
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / passes
    sums = eng.checksum_batch(dec.streams)
    for _, frames in resident:
        for f in frames:
            f.close()
    return ms, frames_per_pass, sums, dec


DUMP_BYTES = 64 * 10**6
DUMP_SEED = 7122


def dump_outputs(out_dir, eng, streams, sums, prefix="", budget=DUMP_BYTES):
    """After the last timed step every stream holds the last frame it decoded; a caller reads it back as cropped
    I420 (read_batch_packed).  Writes, at most `budget` bytes in all, each name preceded by `prefix`:
      last_frame_checksums.npy : float64 (S, 2), the engine's 64-bit checksum of each stream's whole frame as its
                                 high and low 32 bits
      last_frame_samples.npy   : float32 (S, K), the I420 bytes at K positions of each stream's frame: all of them
                                 when the S frames fit, else a sorted sample drawn with a fixed seed
      last_frame_positions.npy : float64 (K,), those byte positions within the I420 frame"""
    import numpy as np
    S = len(streams)
    k = min(FRAME_BYTES, (budget - 16 * S - 3 * 4096) // (4 * S + 8))  # 4096: room for the three .npy headers
    if k == FRAME_BYTES:
        pos = np.arange(FRAME_BYTES)
    else:
        pos = np.sort(np.random.default_rng(DUMP_SEED).choice(FRAME_BYTES, k, replace=False))
    samples = np.empty((S, k), np.float32)
    chunk = 64
    buf = np.empty((chunk, FRAME_BYTES), np.uint8)
    for i in range(0, S, chunk):
        part = streams[i:i + chunk]
        eng.read_batch_packed(part, buf.ctypes.data, FRAME_BYTES)
        samples[i:i + len(part)] = buf[:len(part), pos]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, prefix + "last_frame_checksums.npy"), np.array([[s >> 32, s & 0xFFFFFFFF] for s in sums], np.float64))
    np.save(os.path.join(out_dir, prefix + "last_frame_samples.npy"), samples)
    np.save(os.path.join(out_dir, prefix + "last_frame_positions.npy"), pos.astype(np.float64))


def small_case(torch, dist, world, eng, stream, vp8_b200, payloads, frame_bytes, passes=3):
    """One of the BASELINE configs on this rank's share `payloads` (may be empty).  Returns the whole-job
    kernel-only and end-to-end frames/s (max time over ranks)."""
    n_frames = sum(len(p) for p in payloads)
    k_ms = e_ms = 0.0
    if payloads:
        k_ms, _, sums, dec = kernel_only(torch, eng, stream, vp8_b200, payloads, passes, 2)
        dec.close()
        S = len(payloads)
        e2e = vp8_b200.BatchDecoder(eng, S, parse_threads=max(1, min(S, (os.cpu_count() or 1) // max(1, world))), pinned=True,
                                    tokens_on_device=True, depth=4)
        ring = [torch.empty((S, frame_bytes), dtype=torch.uint8, pin_memory=True) for _ in range(4)]
        packed = (tuple(r.data_ptr() for r in ring), frame_bytes)
        e2e.decode(payloads, out_packed=packed)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(passes):
            e2e.reset()
            e2e.decode(payloads, out_packed=packed)
        torch.cuda.synchronize()
        e_ms = 1e3 * (time.perf_counter() - t0) / passes
        if eng.checksum_batch(e2e.streams) != sums:
            raise SystemExit("bench: replay and end-to-end pass disagree (small case)")
        e2e.close()
    tot = torch.tensor([k_ms, e_ms, float(n_frames)], device="cuda", dtype=torch.float64)
    if world > 1:
        mx = tot.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = tot.clone()
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        k_ms, e_ms, n_frames = float(mx[0]), float(mx[1]), float(sm[2])
    return {"frames": int(n_frames), "kernel_only_frames_per_s": n_frames / (k_ms / 1e3) if k_ms else None,
            "e2e_frames_per_s": n_frames / (e_ms / 1e3) if e_ms else None}


def d2h_ceiling(torch, dist, world, bytes_per_step, reps=6):
    """What the box lets through when every rank does nothing but the read-back of one step (pinned
    destination, all ranks at once): the ceiling of any end-to-end number that delivers full frames."""
    n = max(1, int(bytes_per_step))
    src = torch.empty(n, dtype=torch.uint8, device="cuda")
    dst = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    dst.copy_(src, non_blocking=True)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        dst.copy_(src, non_blocking=True)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([dt], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    del src, dst
    return reps * n / dt  # bytes per second and rank


def parity_against_reference(eng, vp8_b200, torch, payloads, ref_md5s, device_share):
    """Streams 0..P-1 of the workload through the public API (same parse mix as the end-to-end pass): MD5 of
    every shown frame against what the reference decoder wrote for the same stream."""
    P = len(ref_md5s)
    dec = vp8_b200.BatchDecoder(eng, P, parse_threads=min(P, os.cpu_count() or 1), pinned=True, device_parse=device_share, depth=2)
    out = torch.empty((P, FRAME_BYTES), dtype=torch.uint8, pin_memory=True)
    got = [[] for _ in range(P)]
    everyone = list(range(P))
    for t in range(FRAMES):
        frames = dec.parse_step(t % 2, [p[t] for p in payloads[:P]], everyone)
        eng.reconstruct_batch(dec.streams, frames)
        eng.read_batch_packed(dec.streams, out.data_ptr(), FRAME_BYTES, async_=False)
        eng.sync()
        for k, f in enumerate(frames):
            if f.desc().hdr.show_frame:
                got[k].append(hashlib.md5(out[k].numpy().tobytes()).hexdigest())
    dec.close()
    frames = sum(len(g) for g in got)
    bad = [(k, i) for k in range(P) for i in range(max(len(got[k]), len(ref_md5s[k])))
           if i >= len(got[k]) or i >= len(ref_md5s[k]) or got[k][i] != ref_md5s[k][i]]
    return {"streams": P, "frames": frames, "ok": not bad, "first_mismatch": bad[0] if bad else None,
            "against": "oracle/_ref (the unmodified reference decoder), MD5 per shown frame"}


def secondary_roofline(value_frames_per_s, world, sm_mhz):
    """Instruction issue: warp instructions per frame of the reconstruction kernels (committed ncu capture,
    profiles/ncu_traffic.json) against 148 SMs x 4 warp instructions per clock."""
    try:
        inst = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))["warp_instructions_per_frame"]
    except Exception:
        return None
    per_frame = float(sum(v for v in inst.values() if isinstance(v, (int, float))))
    clock = (sm_mhz or 1965) * 1e6
    peak = 148 * 4 * clock
    achieved = per_frame * value_frames_per_s / max(1, world)
    return {"bound": "issue", "warp_inst_per_frame": per_frame, "by_kernel": inst, "peak_warp_inst_per_s": peak,
            "achieved_warp_inst_per_s": achieved, "frac": achieved / peak}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--streams", type=int, default=512, help="independent 1080p streams per GPU")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the BASELINE config 3/4/5 block")
    ap.add_argument("--e2e-parse", default="device", choices=["host", "tokens", "device", "mix"],
                    help="end-to-end pass: where the bitstream is parsed. host: everything on host threads; tokens: "
                         "first partition on the host, DCT token partitions on the GPU; device: frame headers on the "
                         "host, all per-macroblock syntax on the GPU (default); mix: tokens on the GPU, macroblock "
                         "headers on the GPU for --device-share of the streams and on host threads for the rest")
    ap.add_argument("--device-share", type=float, default=None,
                    help="mix: share of the streams whose macroblock headers are decoded on the GPU "
                         "(default 1 - 0.4/n_gpus: the host cores are shared by all ranks)")
    ap.add_argument("--serial-setup", action="store_true", help="generate the streams one at a time (for runs under ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one left in the streams to DIR/*.npy "
                         "(DIR/rank<r>_*.npy per rank when there are several)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import vp8_b200  # raises when libvp8r.so is missing: there is no fallback
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the reconstruction path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        # NCCL prints its version banner to stdout when the communicator is created: keep stdout for
        # the one JSON line
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    S = args.streams
    stream = torch.cuda.Stream()
    eng = vp8_b200.Engine(local_rank, cuda_stream=stream.cuda_stream)
    eng.set_timing(True)

    # ---- inputs: S synthetic streams for this rank (untimed) ----
    tmp = tempfile.mkdtemp()
    from concurrent.futures import ThreadPoolExecutor
    paths = [os.path.join(tmp, f"s{k}.ivf") for k in range(S)]
    gen_workers = 1 if args.serial_setup else max(1, (os.cpu_count() or 1) // max(1, world))
    with ThreadPoolExecutor(max_workers=gen_workers) as ex:
        list(ex.map(lambda k: synth_stream(7122 + rank * S + k, paths[k]), range(S)))
    payloads = [vp8_b200.read_ivf(p)[1] for p in paths]
    shutil.rmtree(tmp, ignore_errors=True)
    ivf_bytes = sum(len(f) for p in payloads for f in p)

    # ---- kernel-only: parse + upload every frame once, then replay ----
    dec = vp8_b200.BatchDecoder(eng, S, pinned=False)
    resident = []  # resident[t] = frames of time step t
    shown_per_pass = 0
    everyone = list(range(S))
    for t in range(FRAMES):
        frames = dec.parse_into([vp8_b200.ParsedFrame(pinned=False) for _ in range(S)], [p[t] for p in payloads], everyone)
        for f in frames:
            shown_per_pass += f.desc().hdr.show_frame
            eng.upload(f, release_host=True)  # the replay only needs the device copy
        resident.append(frames)

    def device_pass():
        for t in range(FRAMES):
            eng.reconstruct_batch(dec.streams, resident[t])

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        device_pass()
    barrier()
    eng.timers(reset=True)
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        ev0.record(stream)
        for _ in range(args.steps):
            device_pass()
        ev1.record(stream)
    barrier()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop()
    tm = eng.timers(reset=True)
    sums = eng.checksum_batch(dec.streams)  # last frame of every stream, compared below with the e2e pass
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, eng, dec.streams, sums, "" if world == 1 else f"rank{rank}_", DUMP_BYTES // world)
        eng.timers(reset=True)  # the read-back's pack kernels are not part of the end-to-end pass
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    frames_per_step = S * FRAMES
    value = world * frames_per_step * args.steps / (ms / 1e3)

    kern_ms = tm.ms_inter + tm.ms_intra + tm.ms_filter + tm.ms_border
    peak, peak_kind = peak_hbm()
    achieved = tm.alg_bytes / (kern_ms / 1e3) / 1e9 if kern_ms > 0 else 0.0
    shares = {"inter": tm.ms_inter, "intra": tm.ms_intra, "filter": tm.ms_filter, "border": tm.ms_border}
    dominant = max(shares, key=shares.get)
    n_launch = {"inter": tm.launches_inter, "intra": tm.launches_intra, "filter": tm.launches_filter}
    traffic = None
    try:
        per_frame = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))[dominant]["bytes_per_frame"]
        traffic = per_frame * S  # per launch of the dominant kernel (S frames), from the committed ncu capture
    except Exception:
        pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "peak_kind": peak_kind, "dominant_kernel": dominant,
                "kernel_ms": {k: round(v, 3) for k, v in shares.items()},
                "dominant_avg_launch_ms": shares[dominant] / max(1, n_launch[dominant]),
                "alg_bytes_per_frame": tm.alg_bytes / max(1, tm.frames)}
    # per-kernel view: the same algorithmic bytes attributed to the kernel that moves them (the loop filter
    # reads and writes every frame once; motion compensation reads one reference frame, writes the frame
    # and reads the coded coefficients), over that kernel's own device time
    plane_bytes = 1.5 * W * ((H + 15) // 16 * 16)
    n_inter_frames = tm.frames * (FRAMES - 1) / FRAMES
    per_kernel = {}
    for name, alg, ms_k in (("filter", tm.frames * 2 * plane_bytes, tm.ms_filter),
                            ("inter", n_inter_frames * 2 * plane_bytes + 32.0 * tm.coef_blocks, tm.ms_inter)):
        if ms_k > 0:
            a = alg / (ms_k / 1e3) / 1e9
            per_kernel[name] = {"achieved": a, "frac": a / peak, "alg_bytes_per_launch": alg / max(1, n_launch[name]),
                                "avg_launch_ms": ms_k / max(1, n_launch[name])}
    roofline["per_kernel"] = per_kernel
    roofline["secondary"] = secondary_roofline(value, world, clocks.get("sm_mhz"))
    launches = tm.launches_inter + tm.launches_intra + 2 * tm.launches_filter  # one BorderKernel behind every filter launch

    # ---- end to end: compressed frames in host memory -> cropped I420 of the shown frames in pinned host memory ----
    for f in (f for fr in resident for f in fr):
        f.close()
    dec.close()
    device_share = args.device_share if args.device_share is not None else 1.0 - 0.4 / world
    # time steps in flight between host parse and the arrival of the frames in host memory (each holds
    # S x 3.1 MB of pinned output; one step less when several ranks share the host's memory)
    DEPTH = 4 if world == 1 else 3
    parse_mode = {"device": True, "mix": device_share}.get(args.e2e_parse, False)
    e2e_dec = vp8_b200.BatchDecoder(eng, S, parse_threads=max(1, min(S, (os.cpu_count() or 1) // max(1, world))), pinned=True,
                                   tokens_on_device=args.e2e_parse == "tokens", device_parse=parse_mode, depth=DEPTH)
    ring_t = [torch.empty((S, FRAME_BYTES), dtype=torch.uint8, pin_memory=True) for _ in range(DEPTH)]
    packed = (tuple(r.data_ptr() for r in ring_t), FRAME_BYTES)  # device-side crop+pack, one D2H per step
    e2e_dec.decode(payloads, out_packed=packed)  # warm-up (allocations, pinned buffers growth)
    barrier()
    t0 = time.perf_counter()
    for k in range(args.e2e_steps):
        # one set of S streams after another, as a server would be handed them: the next pass starts while the last
        # time steps of this one are still on their way (parse -> reconstruction -> read-back is ~100 ms deep);
        # the last pass drains, and the clock stops after that
        e2e_dec.reset()
        decoded, shown, h2d, d2h = e2e_dec.decode(payloads, out_packed=packed, drain=k + 1 == args.e2e_steps)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    host_seconds = {k: round(v, 3) for k, v in getattr(e2e_dec, "host_seconds", {}).items()}  # last pass, this rank
    e2e_sums = eng.checksum_batch(e2e_dec.streams)
    if e2e_sums != sums:
        raise SystemExit("bench: device-resident replay and end-to-end pass disagree on the final frames")
    if world > 1:
        t = torch.tensor([e2e_s], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_value = world * frames_per_step * args.e2e_steps / e2e_s
    tm2 = eng.timers(reset=True)
    parse_threads = e2e_dec.parse_threads
    e2e_dec.close()
    del ring_t
    ceiling_bps = d2h_ceiling(torch, dist, world, d2h / FRAMES)  # one time step's read-back, all ranks at once
    d2h_ceiling_fps = world * ceiling_bps / (d2h / decoded) if d2h else None

    # ---- CPU baseline (reference decoder on the host cores) and parity of the benched workload against it ----
    cpu = parity = None
    binary, ref_flags = ref_decoder()
    if rank == 0 and world == 1 and not args.no_cpu_baseline and binary:
        cores = min(os.cpu_count() or 1, 64, S)
        with tempfile.TemporaryDirectory() as td:
            n_fr = FRAMES
            cpaths = cpu_sample(cores, n_fr, td)
            dt, ref_md5s = run_reference_cpu(cpaths, cores, keep_md5=True)
        cpu = {"value": cores * n_fr / dt, "unit": "frames/s", "cores": cores, "kind": "reference",
               "sample": f"{cores} synthetic 1080p streams x {n_fr} frames (streams 0..{cores - 1} of the GPU workload), one "
                         f"oracle/_ref/{os.path.basename(binary)} process per core ({ref_flags}), {dt:.1f} s"}
        parity = parity_against_reference(eng, vp8_b200, torch, payloads, ref_md5s, parse_mode)

    # ---- BASELINE configs 3, 4, 5 (untimed with respect to the numbers above) ----
    configs = None
    if not args.no_configs:
        configs = {}
        configs["config3_one_1080p_stream"] = small_case(torch, dist, world, eng, stream, vp8_b200,
                                                         payloads[:1] if rank == 0 else [], FRAME_BYTES)
        # 64 streams in total: global stream g lives on rank g % world (vp8_b200.shard.stream_owner); every rank
        # generated its own seeds above, so it takes its first 64/world of them
        n4 = len(vp8_b200.shard.streams_of_rank(64, rank, world))
        configs["config4_64_streams_total"] = small_case(torch, dist, world, eng, stream, vp8_b200, payloads[:min(n4, S)], FRAME_BYTES)
        configs["config4_64_streams_total"]["streams_per_gpu"] = [len(vp8_b200.shard.streams_of_rank(64, r, world)) for r in range(world)]
        with tempfile.TemporaryDirectory() as td:
            p = os.path.join(td, "uhd.ivf")
            subprocess.check_call([SYNTH] + UHD_ARGS.split() + ["--out", p])
            segs = vp8_b200.shard.split_at_key_frames(vp8_b200.read_ivf(p)[1])
        mine = [s for _, (_, s) in vp8_b200.shard.segments_of_rank(segs, rank, world)]
        configs["config5_2160p_gop_segments"] = small_case(torch, dist, world, eng, stream, vp8_b200, mine, UHD_FRAME_BYTES)
        configs["config5_2160p_gop_segments"]["segments"] = len(segs)
        configs["note"] = ("whole-job frames/s, time = max over ranks; end to end with the DCT tokens decoded on the GPU and "
                           "cropped I420 of every shown frame delivered to pinned host memory")
    eng.close()

    if rank == 0:
        shown_frac = shown_per_pass / frames_per_step
        line = {
            "metric": "decoded 1080p frames/s", "value": value, "unit": "frames/s", "n_gpus": world,
            "value_scope": "reconstruction kernels only, parsed frames resident in HBM; bitstream parse, H2D and read-back "
                           "are in e2e, which is the number to compare with the reference arm",
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": f"{S} independent synthetic 1920x1080 30-frame VP8 streams per GPU (vp8synth seeds 7122+k: "
                                   "1 key + 29 inter frames, six-tap MC, normal loop filter level 24, segmentation, "
                                   "golden/altref updates, 4 DCT partitions), decoded in lock-step batches of one frame per stream",
                       "streams_per_gpu": S, "frames_per_stream": FRAMES, "shown_frames_per_step": shown_per_pass,
                       "mp_per_s": value * shown_frac * W * H / 1e6, "mp_per_s_counts": "shown frames x 1920 x 1080 (SURVEY 8(d))",
                       "compressed_bytes_per_step": ivf_bytes,
                       "l2_policy": "inputs larger than L2 (one batch of %d frames touches ~%d MB of surfaces and side data)" % (S, S * 8),
                       "parse_threads": parse_threads},
            "roofline": roofline,
            "cpu_baseline": cpu,
            "parity_checked": parity,
            "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "mp_per_s": e2e_value * shown_frac * W * H / 1e6, "steps": args.e2e_steps,
                    "shown_frames_per_s": e2e_value * shown_frac,
                    "kernel_ms_per_step": (tm2.ms_inter + tm2.ms_intra + tm2.ms_filter + tm2.ms_border) / max(1, args.e2e_steps + 1),
                    "token_kernel_ms_per_step": tm2.ms_tokens / max(1, args.e2e_steps + 1),
                    "parse": args.e2e_parse, "device_header_share": device_share if args.e2e_parse == "mix" else None,
                    "steps_in_flight": DEPTH, "host_seconds_last_pass": host_seconds,
                    "d2h_ceiling_frames_per_s": d2h_ceiling_fps, "d2h_ceiling_gb_per_s_per_gpu": ceiling_bps / 1e9,
                    "frac_of_d2h_ceiling": e2e_value / d2h_ceiling_fps if d2h_ceiling_fps else None,
                    "limiter": None},
            "configs": configs,
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
        e = line["e2e"]
        if e["frac_of_d2h_ceiling"] and e["frac_of_d2h_ceiling"] > 0.8:
            e["limiter"] = "read-back of full I420 frames into host memory (PCIe / host memory bandwidth shared by the ranks)"
        elif host_seconds.get("parse", 0) > 0.5 * e2e_s / max(1, args.e2e_steps):
            e["limiter"] = "host threads: frame-header / first-partition parse on the cores this rank gets"
        else:
            e["limiter"] = ("device-side parse kernels (one single-lane warp per bool-coded partition: latency-bound chains whose registers "
                            "fill the SMs) sharing the GPU with the reconstruction kernels; read-back at %.0f %% of its ceiling" % (100 * (e["frac_of_d2h_ceiling"] or 0)))
        print(json.dumps(line))
        if parity is not None and not parity["ok"]:
            raise SystemExit("bench: the GPU output differs from the reference decoder on the benched workload")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
