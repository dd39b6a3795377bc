"""Host-side mirror of the reference's decode loop (src/decode.cc:50-77) over the C ABI.

    Parser        <-> BitstreamParser + ParserContext       (host only)
    Engine/Stream <-> DecodeFrame + RefreshRefFrames + YUV::WriteFrame on the GPU

There is no CPU implementation of the pixel path here: Engine() raises when libvp8r.so is missing
or no sm_100 GPU is visible.
"""
import ctypes as C

from . import _capi
from ._capi import check


DEVICE_LAYOUTS = {"i420": 0, "nv12": 1, "rgb": 2, "rgb_planar": 3}  # VP8R_LAYOUT_*
ENC_BPRED, ENC_INTRA_MBS = 1, 2  # VP8R_ENC_BPRED, VP8R_ENC_INTRA_MBS


def _is_tensor(x):
    """A torch.Tensor, without importing torch for callers that never pass one."""
    return type(x).__module__.startswith("torch") and hasattr(x, "data_ptr")


def _layout_bytes(stream, layout):
    """Bytes of the stream's latest frame in a device read-back layout (0 before its first frame)."""
    if layout in ("i420", "nv12") or stream.frame_bytes() == 0:
        return stream.frame_bytes()
    w, h = stream.dims()
    return 3 * w * h


class ParsedFrame:
    def __init__(self, pinned=False):
        self._lib = _capi.load()
        self.handle = self._lib.vp8r_frame_create(1 if pinned else 0)
        if not self.handle:
            raise MemoryError("vp8r_frame_create")

    def desc(self):
        d = _capi.FrameDesc()
        check(self._lib.vp8r_frame_get_desc(self.handle, C.byref(d)))
        return d

    def write_bitstream(self, context=None):
        """The frame as a VP8 frame, key or inter (the inverse of Parser.parse for what the encoder produces; see
        vp8r_frame_write_bitstream for the frames that can be written).  context: the Parser that parsed the stream so
        far; an inter frame is then coded with that stream's current probabilities instead of the defaults, which it
        must be when the stream's LAST frame came from decoding (vp8r_frame_write_bitstream_in)."""
        ctx = context.handle if context is not None else None
        size = C.c_size_t(0)
        rc = self._lib.vp8r_frame_write_bitstream_in(self.handle, ctx, None, 0, C.byref(size))
        if size.value == 0:
            check(rc)
        buf = (C.c_uint8 * size.value)()
        check(self._lib.vp8r_frame_write_bitstream_in(self.handle, ctx, buf, size.value, C.byref(size)))
        return bytes(buf[:size.value])

    def close(self):
        if self.handle:
            self._lib.vp8r_frame_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Parser:
    """One per stream: carries probability / segmentation state between frames."""

    def __init__(self):
        self._lib = _capi.load()
        self.handle = self._lib.vp8r_parser_create()

    def parse(self, payload, out=None, pinned=False):
        out = out or ParsedFrame(pinned=pinned)
        buf = (C.c_uint8 * len(payload)).from_buffer_copy(payload) if len(payload) else (C.c_uint8 * 1)()
        check(self._lib.vp8r_parser_parse(self.handle, buf, len(payload), out.handle))
        return out

    def reset(self):
        self._lib.vp8r_parser_reset(self.handle)

    def set_defer_tokens(self, on=True):
        """First partition only on the host; the DCT partitions travel with the frame and are
        decoded by the engine's token kernel (vp8r_frame_hdr.tokens_deferred)."""
        self._lib.vp8r_parser_set_defer_tokens(self.handle, 1 if on else 0)

    def set_defer_modes(self, on=True):
        """Frame headers only on the host; the per-macroblock syntax of the first partition and the
        DCT partitions are decoded by the engine's parse kernel (vp8r_frame_hdr.modes_deferred)."""
        self._lib.vp8r_parser_set_defer_modes(self.handle, 1 if on else 0)

    def close(self):
        if self.handle:
            self._lib.vp8r_parser_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Engine:
    def __init__(self, device=0, cuda_stream=None):
        self._lib = _capi.load()
        h = C.c_void_p()
        check(self._lib.vp8r_engine_create(device, C.c_void_p(cuda_stream) if cuda_stream else None, C.byref(h)))
        self.handle = h
        self.device = device

    def open_stream(self):
        return Stream(self)

    def reconstruct_batch(self, streams, frames):
        n = len(streams)
        sa = (C.c_void_p * n)(*[s.handle for s in streams])
        fa = (C.c_void_p * n)(*[f.handle for f in frames])
        check(self._lib.vp8r_reconstruct_batch(self.handle, n, sa, fa))

    def encode_key_frames(self, streams, images, width, height, q_index, loop_filter_level=0, sharpness=0, bpred=True,
                          layout="i420"):
        """Row f4: one key frame per stream from cropped I420 images (bytes), encoded in a closed loop on the device.
        Returns the ParsedFrame objects (macroblock records + coefficient blocks; .write_bitstream() serialises them);
        every stream then holds the reconstructed frame a decoder would produce.  bpred: B_PRED (sixteen 4x4 modes per
        macroblock) competes with the four 16x16 modes (VP8R_ENC_BPRED).  `images` may instead be a contiguous
        torch.uint8 CUDA tensor on the engine's device with one frame per stream along its first dimension, in `layout`
        (see _device_source); it is read on the device, ordered behind the work queued on torch's current stream."""
        return self._encode(self._lib.vp8r_encode_key_frames, self._lib.vp8r_encode_key_frames_device, streams, images,
                            layout, width, height, q_index, loop_filter_level, sharpness, ENC_BPRED if bpred else 0)

    def encode_inter_frames(self, streams, images, width, height, q_index, loop_filter_level=0, sharpness=0, search_range=16,
                            layout="i420", intra_mbs=False, bpred=True):
        """One inter frame per stream from cropped I420 images (bytes): every macroblock predicts from the stream's
        current LAST frame with one motion vector, searched on the device over +-search_range whole pixels (4..24) and
        refined to quarter pel (vp8r_encode_inter_frames_ex).  intra_mbs: a macroblock that LAST predicts worse than
        intra prediction does, by more than a bias of the quantiser, is coded intra instead (VP8R_ENC_INTRA_MBS), with
        B_PRED among its candidates when bpred is set (VP8R_ENC_BPRED); bpred is ignored without intra_mbs.  Returns the
        ParsedFrame objects (records with modes and vectors, coefficient blocks; .write_bitstream() serialises them);
        every stream then holds the reconstructed frame a decoder would produce.  `images` and `layout` as for
        encode_key_frames."""
        flags = (ENC_INTRA_MBS | (ENC_BPRED if bpred else 0)) if intra_mbs else 0
        return self._encode(self._lib.vp8r_encode_inter_frames_ex, self._lib.vp8r_encode_inter_frames_device_ex, streams,
                            images, layout, width, height, q_index, loop_filter_level, sharpness, search_range, flags)

    def _encode(self, fn, fn_device, streams, images, layout, width, height, *params):
        """Calls the C encoder entry point on one picture per stream: fn(engine, n, streams, images, width, height,
        *params, frames) for cropped I420 images (bytes), fn_device(engine, n, streams, src, stride, layout, producer,
        width, height, *params, frames) for a CUDA tensor; returns the new ParsedFrame objects."""
        n = len(streams)
        if _is_tensor(images):
            src, stride, code, producer = self._device_source(images, n, layout, width, height)
            frames = [ParsedFrame(pinned=False) for _ in range(n)]
            sa = (C.c_void_p * n)(*[s.handle for s in streams])
            fa = (C.c_void_p * n)(*[f.handle for f in frames])
            check(fn_device(self.handle, n, sa, C.c_void_p(src), stride, code, C.c_void_p(producer), width, height, *params,
                            fa))
            return frames
        if layout != "i420":
            raise ValueError(f"layout {layout!r} needs a CUDA tensor: images in host memory are cropped I420 bytes")
        need = width * height + 2 * ((width + 1) // 2) * ((height + 1) // 2)
        bufs = []
        for img in images:
            if len(img) != need:
                raise ValueError("image is not a cropped I420 frame of the given size")
            bufs.append((C.c_uint8 * need).from_buffer_copy(img))
        frames = [ParsedFrame(pinned=False) for _ in range(n)]
        sa = (C.c_void_p * n)(*[s.handle for s in streams])
        ia = (C.c_void_p * n)(*[C.cast(b, C.c_void_p) for b in bufs])
        fa = (C.c_void_p * n)(*[f.handle for f in frames])
        check(fn(self.handle, n, sa, ia, width, height, *params, fa))
        return frames

    def _device_source(self, src, n, layout, width, height):
        """Checks a tensor of n source frames: torch.uint8, contiguous, on the engine's device, of shape (n, frame bytes)
        for "i420" / "nv12", (n, H, W, 3) for "rgb", (n, 3, H, W) for "rgb_planar".  Returns (address, stride, layout
        code, producer stream): the producer is torch's current stream, named by cudaStreamLegacy (1) when it is the
        default stream, whose handle 0 the C calls read as "no stream"."""
        import torch
        if layout not in DEVICE_LAYOUTS:
            raise ValueError(f"unknown layout {layout!r}: one of {sorted(DEVICE_LAYOUTS)}")
        if src.dtype != torch.uint8:
            raise ValueError("source tensor must be torch.uint8")
        if src.device != torch.device("cuda", self.device):
            raise ValueError(f"source tensor is on {src.device}, the engine on cuda:{self.device}")
        if not src.is_contiguous():
            raise ValueError("source tensor must be contiguous")
        shape = {"rgb": (height, width, 3), "rgb_planar": (3, height, width)}.get(
            layout, (width * height + 2 * ((width + 1) // 2) * ((height + 1) // 2),))
        if tuple(src.shape) != (n,) + shape:
            raise ValueError(f"source tensor has shape {tuple(src.shape)}, {layout} frames of {width}x{height} for {n} "
                             f"streams need {(n,) + shape}")
        producer = torch.cuda.current_stream(src.device).cuda_stream or 1
        return src.data_ptr(), src[0].numel(), DEVICE_LAYOUTS[layout], producer

    def convert_to_i420(self, src, layout, width, height):
        """The cropped I420 images the encoder codes for a CUDA tensor of n frames in `layout` (as encode_key_frames
        takes it): returns an (n, frame bytes) torch.uint8 CUDA tensor, computed on torch's current stream's order
        (vp8r_convert_to_i420_device)."""
        import torch
        n = src.shape[0] if src.dim() else 0
        s, stride, code, stream = self._device_source(src, n, layout, width, height)
        fb = width * height + 2 * ((width + 1) // 2) * ((height + 1) // 2)
        out = torch.empty((n, fb), dtype=torch.uint8, device=src.device)
        if n:
            check(self._lib.vp8r_convert_to_i420_device(self.handle, n, C.c_void_p(s), stride, code, width, height,
                                                        C.c_void_p(out.data_ptr()), fb, C.c_void_p(stream)))
        return out

    def upload(self, frame, release_host=False):
        """Copies the frame's arrays to HBM; release_host frees the host copy afterwards."""
        check(self._lib.vp8r_frame_upload(self.handle, frame.handle))
        if release_host:
            check(self._lib.vp8r_frame_release_host(frame.handle))

    def checksum_batch(self, streams):
        n = len(streams)
        sa = (C.c_void_p * n)(*[s.handle for s in streams])
        out = (C.c_uint64 * n)()
        check(self._lib.vp8r_checksum_batch(self.handle, n, sa, out))
        return list(out)

    def read_batch(self, streams, ptrs, caps, async_=False):
        n = len(streams)
        sa = (C.c_void_p * n)(*[s.handle for s in streams])
        pa = (C.c_void_p * n)(*ptrs)
        ca = (C.c_size_t * n)(*caps)
        check(self._lib.vp8r_read_batch(self.handle, n, sa, pa, ca, 1 if async_ else 0))

    def read_batch_packed(self, streams, dst_ptr, stride, async_=False, layout="i420"):
        """Device-side crop + pack of every stream's latest frame, one contiguous D2H copy:
        frame i at dst_ptr + i*stride.  layout: "i420" (Y, U, V planes) or "nv12" (Y, interleaved UV)."""
        n = len(streams)
        sa = (C.c_void_p * n)(*[s.handle for s in streams])
        check(self._lib.vp8r_read_batch_packed_as(self.handle, n, sa, C.c_void_p(dst_ptr), stride, 1 if async_ else 0,
                                                  {"i420": 0, "nv12": 1}[layout]))

    def read_batch_device(self, streams, out, layout="rgb"):
        """Every stream's latest frame into row i of `out`, a contiguous torch.uint8 CUDA tensor on the engine's device
        (first dimension >= len(streams), each row at least one frame of the layout).  layout: "i420" or "nv12" (the
        bytes of the packed read-back), "rgb" (BT.601 R,G,B per pixel: rows of shape (H, W, 3)) or "rgb_planar"
        ((3, H, W)).  Asynchronous and ordered against torch's current stream: the conversion waits for the work
        already queued there, and work queued there afterwards sees the frames."""
        import torch
        if layout not in DEVICE_LAYOUTS:
            raise ValueError(f"unknown layout {layout!r}: one of {sorted(DEVICE_LAYOUTS)}")
        n = len(streams)
        if not isinstance(out, torch.Tensor) or out.dtype != torch.uint8:
            raise ValueError("out must be a torch.uint8 tensor")
        if out.device != torch.device("cuda", self.device):
            raise ValueError(f"out is on {out.device}, the engine on cuda:{self.device}")
        if out.dim() < 2 or not out.is_contiguous():
            raise ValueError("out must be a contiguous tensor with one frame per row of its first dimension")
        if out.shape[0] < n:
            raise ValueError(f"out has {out.shape[0]} rows for {n} streams")
        row = out[0].numel() if out.shape[0] else 0  # = out.stride(0), except for one row, whose stride may exceed it
        need = max((_layout_bytes(s, layout) for s in streams), default=0)
        if row < need:
            raise ValueError(f"a row of out holds {row} bytes, a frame needs {need}")
        sa = (C.c_void_p * n)(*[s.handle for s in streams])
        # torch's default stream has the handle 0, which the C call reads as "no consumer stream": name it by
        # cudaStreamLegacy (1) so that the ordering holds for it too
        consumer = torch.cuda.current_stream(out.device).cuda_stream or 1
        check(self._lib.vp8r_read_batch_device(self.handle, n, sa, C.c_void_p(out.data_ptr()), row,
                                               DEVICE_LAYOUTS[layout], C.c_void_p(consumer)))

    def sync(self):
        check(self._lib.vp8r_engine_sync(self.handle))

    def set_timing(self, on):
        check(self._lib.vp8r_engine_set_timing(self.handle, 1 if on else 0))

    def timers(self, reset=False):
        t = _capi.Timers()
        check(self._lib.vp8r_engine_get_timers(self.handle, C.byref(t), 1 if reset else 0))
        return t

    def close(self):
        if self.handle:
            self._lib.vp8r_engine_destroy(self.handle)
            self.handle = None


class Stream:
    """One decoder instance: parser state + last/golden/altref surfaces resident in HBM."""

    def __init__(self, engine):
        self.engine = engine
        self._lib = engine._lib
        h = C.c_void_p()
        check(self._lib.vp8r_stream_open(engine.handle, C.byref(h)))
        self.handle = h

    def decode(self, payload):
        """One iteration of src/decode.cc:50-77.  Returns show_frame."""
        shown = C.c_int(0)
        buf = (C.c_uint8 * max(len(payload), 1)).from_buffer_copy(payload or b"\0")
        check(self._lib.vp8r_stream_decode(self.handle, buf, len(payload), C.byref(shown)))
        return bool(shown.value)

    def frame_bytes(self):
        return self._lib.vp8r_stream_frame_bytes(self.handle)

    def dims(self):
        w, h = C.c_int(), C.c_int()
        check(self._lib.vp8r_stream_dims(self.handle, C.byref(w), C.byref(h)))
        return w.value, h.value

    def read_frame(self):
        n = self.frame_bytes()
        buf = (C.c_uint8 * n)()
        check(self._lib.vp8r_stream_read_frame(self.handle, buf, n))
        return bytes(buf)

    def checksum(self):
        out = C.c_uint64()
        check(self._lib.vp8r_stream_checksum(self.handle, C.byref(out)))
        return out.value

    def close(self):
        if self.handle:
            self._lib.vp8r_stream_close(self.handle)
            self.handle = None


def decode_ivf(path_or_bytes, engine=None, layout=None):
    """`./decode in.ivf out.yuv` (src/decode.cc:13-79): returns the shown frames as I420 bytes.  With a device read-back
    layout ("i420", "nv12", "rgb", "rgb_planar", see Engine.read_batch_device) it returns instead one uint8 CUDA tensor
    of all shown frames on the engine's device: (T, frame bytes) for "i420" / "nv12", (T, H, W, 3) for "rgb",
    (T, 3, H, W) for "rgb_planar".  A stream that changes its size is refused there (ValueError)."""
    from .ivf import read_ivf
    if layout is not None and layout not in DEVICE_LAYOUTS:
        raise ValueError(f"unknown layout {layout!r}: one of {sorted(DEVICE_LAYOUTS)}")
    own = engine is None
    engine = engine or Engine()
    _, payloads = read_ivf(path_or_bytes)
    st = engine.open_stream()
    out, dims = [], None
    try:
        for p in payloads:
            if not st.decode(p):
                continue
            if layout is None:
                out.append(st.read_frame())
                continue
            if dims is None:
                import torch
                dims = st.dims()
                w, h = dims
                shape = {"rgb": (h, w, 3), "rgb_planar": (3, h, w)}.get(layout, (st.frame_bytes(),))
                frames = torch.empty((len(payloads),) + shape, dtype=torch.uint8, device=torch.device("cuda", engine.device))
            elif st.dims() != dims:
                raise ValueError(f"the stream changes its size from {dims} to {st.dims()}: one tensor cannot hold it")
            engine.read_batch_device([st], frames[len(out):len(out) + 1], layout)
            out.append(None)
    finally:
        st.close()
        if own:
            engine.close()
    if layout is None:
        return out
    if dims is None:
        raise ValueError("the stream has no shown frame")
    return frames[:len(out)]


def encode_ivf(images, width, height, q_index, path=None, key_interval=0, loop_filter_level=0, sharpness=0, bpred=True,
               search_range=16, engine=None, layout="i420", intra_mbs=False):
    """Encodes one stream of cropped I420 images (bytes) into an IVF file, the mirror of decode_ivf: a key frame first
    and then every key_interval frames (0: only the first), inter frames between them.  intra_mbs: the inter frames
    may code macroblocks intra where LAST predicts them badly (see Engine.encode_inter_frames); bpred then applies to
    those macroblocks as well.  Returns the IVF bytes and
    writes them to `path` when one is given.  `images` may instead be a (T, ...) torch.uint8 CUDA tensor of T frames in
    `layout` (see Engine.encode_key_frames), such as decode_ivf(..., layout="i420") returns: no pixel then crosses PCIe."""
    from .ivf import ivf_bytes
    if key_interval < 0:
        raise ValueError("key_interval must be >= 0")
    own = engine is None
    engine = engine or Engine()
    st = engine.open_stream()
    payloads = []
    try:
        pictures = (images[i:i + 1] for i in range(len(images))) if _is_tensor(images) else ([img] for img in images)
        for i, img in enumerate(pictures):
            if i == 0 or (key_interval and i % key_interval == 0):
                (f,) = engine.encode_key_frames([st], img, width, height, q_index, loop_filter_level, sharpness, bpred,
                                                layout=layout)
            else:
                (f,) = engine.encode_inter_frames([st], img, width, height, q_index, loop_filter_level, sharpness,
                                                  search_range, layout=layout, intra_mbs=intra_mbs, bpred=bpred)
            payloads.append(f.write_bitstream())
            f.close()
    finally:
        st.close()
        if own:
            engine.close()
    data = ivf_bytes(width, height, payloads)
    if path is not None:
        with open(path, "wb") as fh:
            fh.write(data)
    return data
