"""Lock-step decoding of many independent streams: the throughput-oriented public API.

All streams advance one frame per time step; the frames of one time step are parsed on host
threads (vp8r_parse_batch), reconstructed by one batched launch per kernel class
(vp8r_reconstruct_batch) and, optionally, copied back as cropped I420 (vp8r_read_batch).  Host
parsing of step t+1 overlaps the device work of step t; fences guard the reuse of pinned buffers.
"""
import ctypes as C
import os
import time

from . import _capi
from ._capi import check
from .decoder import ParsedFrame, Parser


class BatchDecoder:
    def __init__(self, engine, n_streams, parse_threads=None, pinned=True, tokens_on_device=False, device_parse=False,
                 depth=2):
        """depth: time steps in flight (parsed-frame slots; out_ring / out_packed passed to decode()
        must hold as many buffers).  The engine supports up to 8."""
        self.engine = engine
        self._lib = engine._lib
        self.n = n_streams
        self.parse_threads = parse_threads or min(n_streams, os.cpu_count() or 1)
        self.parsers = [Parser() for _ in range(n_streams)]
        self.tokens_on_device = tokens_on_device
        self.device_parse = device_parse
        if tokens_on_device:  # host: headers, modes, motion vectors; device: DCT token partitions
            for p in self.parsers:
                p.set_defer_tokens(True)
        if device_parse:      # host: frame headers only; device: all per-macroblock syntax
            # device_parse may be a fraction: that share of the streams has its macroblock headers
            # decoded on the device, the rest on host threads (both feed the same batched launches),
            # which balances the host cores against the GPU's header threads
            share = 1.0 if device_parse is True else float(device_parse)
            n_dev = int(round(share * n_streams))
            for k, p in enumerate(self.parsers):
                if k < n_dev:
                    p.set_defer_modes(True)
                else:
                    p.set_defer_tokens(True)
        self.streams = [engine.open_stream() for _ in range(n_streams)]
        self.depth = max(2, min(8, depth))
        self._g = 0          # time steps submitted so far, over all decode() calls: slot / ring entry = step % depth
        self._tickets = {}   # step -> fence ticket of its kernels and read-back
        self.slots = [[ParsedFrame(pinned=pinned) for _ in range(n_streams)] for _ in range(self.depth)]

    def reset(self):
        for p in self.parsers:
            p.reset()

    @staticmethod
    def _payload_pointers(payloads, live):
        """Array of pointers to the compressed frames.  `bytes` objects are passed in place (the parser
        only reads them during the call); anything else is copied into a ctypes buffer first.  Returns
        (pointer array, objects to keep alive until the call returns)."""
        keep, ptrs = [], []
        for i in live:
            p = payloads[i]
            if isinstance(p, bytes):
                ptrs.append(C.cast(C.c_char_p(p), C.c_void_p))
            else:
                buf = (C.c_uint8 * max(len(p), 1)).from_buffer_copy(bytes(p) or b"\0")
                keep.append(buf)
                ptrs.append(C.cast(buf, C.c_void_p))
        return (C.c_void_p * len(ptrs))(*ptrs), keep

    def parse_step(self, slot, payloads, live):
        """Parses payloads[i] (bytes) of the live streams into slot `slot`.  Returns the frames."""
        n = len(live)
        pa = (C.c_void_p * n)(*[self.parsers[i].handle for i in live])
        da, keep = self._payload_pointers(payloads, live)
        sa = (C.c_size_t * n)(*[len(payloads[i]) for i in live])
        frames = [self.slots[slot][i] for i in live]
        fa = (C.c_void_p * n)(*[f.handle for f in frames])
        check(self._lib.vp8r_parse_batch(n, pa, da, sa, fa, self.parse_threads, None))
        return frames

    def parse_into(self, frames, payloads, live):
        """Parses payloads[i] of the live streams into caller-owned ParsedFrame objects (host threads)."""
        n = len(live)
        pa = (C.c_void_p * n)(*[self.parsers[i].handle for i in live])
        da, keep = self._payload_pointers(payloads, live)
        sa = (C.c_size_t * n)(*[len(payloads[i]) for i in live])
        fa = (C.c_void_p * n)(*[f.handle for f in frames])
        check(self._lib.vp8r_parse_batch(n, pa, da, sa, fa, self.parse_threads, None))
        return frames

    def fence(self):
        t = C.c_uint64()
        check(self._lib.vp8r_engine_fence(self.engine.handle, C.byref(t)))
        return t.value

    def wait(self, ticket):
        check(self._lib.vp8r_engine_wait(self.engine.handle, ticket))

    def decode(self, payloads, out_ring=None, on_step=None, out_packed=None, shown_only=True, drain=True, out_device=None):
        """payloads[s] = list of compressed frames of stream s.  out_ring: optional list of `depth` lists
        of (ptr, capacity) pinned host buffers, one per stream, that receive the frames of a time step
        (ring of `depth` steps).  out_packed: optional ((ptr0, ptr1, ...), stride): `depth` pinned host
        buffers; the frames of a time step are cropped and packed on the device and arrive with one copy,
        frame k of the step's live streams at ptr + k*stride.  shown_only (default): only frames with
        show_frame set are read back (the reference never writes a hidden frame, src/decode.cc:76), so frame k
        of the packed buffer is the k-th SHOWN frame of the step.  on_step(t, live, frames) is called after
        step t has been submitted.  drain=False returns without waiting for the last steps: the next decode()
        (new streams after reset(), same rings) then starts while they finish, as a server that is handed one set
        of streams after another would run; the ring entry of a step is (steps since the last drain) % depth, and the
        last call has to drain (or the caller calls engine.sync()).
        out_device: optional (ring, layout): `depth` uint8 CUDA tensors on the engine's device; the frames of a time
        step stay on the GPU, frame k of the step in row k of its ring entry (same indexing as out_packed), in `layout`
        ("i420", "nv12", "rgb" or "rgb_planar", Engine.read_batch_device), ordered against torch's current stream.
        These bytes do not count as d2h.  out_packed and out_device may be given together.
        Returns (frames decoded, frames shown, h2d bytes, d2h bytes)."""
        steps = max(len(p) for p in payloads)
        decoded = shown = h2d = d2h = 0
        self.host_seconds = {"parse": 0.0, "submit": 0.0, "readback": 0.0, "wait": 0.0, "account": 0.0}
        hs, clock = self.host_seconds, time.perf_counter
        tickets, g0, depth = self._tickets, self._g, self.depth
        live = [i for i in range(self.n) if len(payloads[i]) > 0]
        t0 = clock()
        if g0 - depth in tickets:
            self.wait(tickets.pop(g0 - depth))
        hs["wait"] += clock() - t0
        t0 = clock()
        frames = self.parse_step(g0 % depth, [p[0] if p else b"" for p in payloads], live)
        hs["parse"] += clock() - t0
        for t in range(steps):
            g = g0 + t
            t0 = clock()
            streams = [self.streams[i] for i in live]
            self.engine.reconstruct_batch(streams, frames)
            hs["submit"] += clock() - t0
            t0 = clock()
            decoded += len(live)
            out_idx = []
            for k, f in enumerate(frames):
                d = f.desc()
                h2d += (0 if d.hdr.modes_deferred else d.hdr.mb_cols * d.hdr.mb_rows * 32) + d.hdr.n_payload_blocks * 32
                shown += d.hdr.show_frame
                if d.hdr.show_frame or not shown_only:
                    out_idx.append(k)
            hs["account"] += clock() - t0
            t0 = clock()
            if out_ring is not None and out_idx:
                ring = out_ring[g % depth]
                self.engine.read_batch([streams[k] for k in out_idx], [ring[live[k]][0] for k in out_idx],
                                       [ring[live[k]][1] for k in out_idx], async_=True)
                d2h += sum(streams[k].frame_bytes() for k in out_idx)
            if out_packed is not None and out_idx:
                (ptrs, stride) = out_packed
                self.engine.read_batch_packed([streams[k] for k in out_idx], ptrs[g % depth], stride, async_=True)
                d2h += len(out_idx) * stride
            if out_device is not None and out_idx:
                ring, layout = out_device
                self.engine.read_batch_device([streams[k] for k in out_idx], ring[g % depth], layout)
            tickets[g] = self.fence()
            hs["readback"] += clock() - t0
            if on_step:
                on_step(t, live, frames)
            if t + 1 < steps:
                old = g + 1 - depth
                t0 = clock()
                if old in tickets:
                    self.wait(tickets.pop(old))  # slot and ring entry (g+1) % depth are free again
                hs["wait"] += clock() - t0
                t0 = clock()
                live = [i for i in range(self.n) if len(payloads[i]) > t + 1]
                frames = self.parse_step((g + 1) % depth, [p[t + 1] if len(p) > t + 1 else b"" for p in payloads], live)
                hs["parse"] += clock() - t0
        self._g = g0 + steps
        if drain:
            self.engine.sync()
            tickets.clear()
            self._g = 0
        return decoded, shown, h2d, d2h

    def close(self):
        for s in self.streams:
            s.close()
        for p in self.parsers:
            p.close()
        for sl in self.slots:
            for f in sl:
                f.close()
