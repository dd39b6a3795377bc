"""Encoder input from device memory (vp8r_encode_key_frames_device, vp8r_encode_inter_frames_device,
vp8r_convert_to_i420_device; Engine.encode_*_frames / convert_to_i420 / encode_ivf with a CUDA tensor).  CPU tier: the
numpy BT.601 RGB -> I420 reference below and the argument checks that need no device.  GPU tier: the conversion equals
that reference bit for bit in every layout, and every layout encodes exactly what the host path encodes for its I420
image: the same records, coefficient blocks, bitstream and reconstruction."""
import ctypes as C
import os

import numpy as np
import pytest

import helpers

VP8R_ERR_INVALID_ARG = 1
LAYOUTS = ("i420", "nv12", "rgb", "rgb_planar")


# ---- reference conversion: BT.601 limited range in integers, include/vp8r.h -----------------------------------------
def rgb_to_i420(rgb):
    """(h, w, 3) uint8 RGB -> cropped I420 bytes.  Y per pixel; U, V per chroma sample from the channel means
    (s + 2) >> 2 of its 2x2 pixels, pixel coordinates clamped to w-1 / h-1."""
    a = rgb.astype(np.int32)
    h, w = a.shape[:2]
    y = ((66 * a[..., 0] + 129 * a[..., 1] + 25 * a[..., 2] + 128) >> 8) + 16
    cw, ch = (w + 1) // 2, (h + 1) // 2
    p = a[np.minimum(np.arange(2 * ch), h - 1)][:, np.minimum(np.arange(2 * cw), w - 1)]
    m = (p[0::2, 0::2] + p[0::2, 1::2] + p[1::2, 0::2] + p[1::2, 1::2] + 2) >> 2
    u = ((-38 * m[..., 0] - 74 * m[..., 1] + 112 * m[..., 2] + 128) >> 8) + 128
    v = ((112 * m[..., 0] - 94 * m[..., 1] - 18 * m[..., 2] + 128) >> 8) + 128
    return np.concatenate([y.ravel(), u.ravel(), v.ravel()]).astype(np.uint8).tobytes()


def i420_to_nv12(img, w, h):
    cn = ((w + 1) // 2) * ((h + 1) // 2)
    a = np.frombuffer(img, np.uint8)
    return a[:w * h].tobytes() + np.stack([a[w * h:w * h + cn], a[w * h + cn:]], axis=1).tobytes()


def source_frame(layout, w, h, seed):
    """A seeded frame in `layout` (numpy uint8, the shape the tensor API takes per frame) and its cropped I420 bytes."""
    rng = np.random.default_rng(seed)
    if layout in ("i420", "nv12"):
        img = rng.integers(0, 256, helpers.i420_bytes(w, h), dtype=np.uint8).tobytes()
        data = img if layout == "i420" else i420_to_nv12(img, w, h)
        return np.frombuffer(data, np.uint8).copy(), img
    rgb = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    img = rgb_to_i420(rgb)
    return (rgb if layout == "rgb" else np.ascontiguousarray(rgb.transpose(2, 0, 1))), img


# ---- CPU tier --------------------------------------------------------------------------------------------------------
def _all_triples(r):
    g, b = np.meshgrid(np.arange(256), np.arange(256), indexing="ij")
    return np.stack([np.full(65536, r), g.ravel(), b.ravel()], axis=-1)


def test_reference_within_one_of_float_bt601_and_in_range():
    """Every (R, G, B) as a uniform 2x2 block (so the chroma means are the pixel): Y, U, V within 1 of the rounded
    floating-point BT.601 limited-range matrix, Y in 16..235, U and V in 16..240."""
    worst, lo, hi = 0, np.array([255] * 3), np.array([0] * 3)
    for r in range(256):
        t = _all_triples(r)
        block = np.repeat(np.repeat(t.reshape(256, 256, 1, 1, 3), 2, axis=2), 2, axis=3)  # (g, b, 2, 2, 3)
        img = block.transpose(0, 2, 1, 3, 4).reshape(512, 512, 3)
        out = np.frombuffer(rgb_to_i420(img.astype(np.uint8)), np.uint8).astype(np.int32)
        y = out[:512 * 512].reshape(512, 512)[0::2, 0::2].ravel()
        u = out[512 * 512:512 * 512 + 65536]
        v = out[512 * 512 + 65536:]
        R, G, B = (t[:, k].astype(np.float64) for k in range(3))
        fy = 16 + 219 * (0.299 * R + 0.587 * G + 0.114 * B) / 255
        fu = 128 + 224 * (-0.168736 * R - 0.331264 * G + 0.5 * B) / 255
        fv = 128 + 224 * (0.5 * R - 0.418688 * G - 0.081312 * B) / 255
        got = np.stack([y, u, v], axis=-1)
        ref = np.rint(np.stack([fy, fu, fv], axis=-1))
        worst = max(worst, int(np.abs(got - ref).max()))
        lo, hi = np.minimum(lo, got.min(axis=0)), np.maximum(hi, got.max(axis=0))
    assert worst <= 1, worst
    assert tuple(lo) >= (16, 16, 16) and tuple(hi) <= (235, 240, 240), (lo, hi)


def test_reference_pinned_values():
    pts = {(0, 0, 0): (16, 128, 128), (255, 255, 255): (235, 128, 128), (128, 128, 128): (126, 128, 128),
           (255, 0, 0): (82, 90, 240), (0, 255, 0): (144, 54, 34), (0, 0, 255): (41, 240, 110)}
    for rgb, want in pts.items():
        assert tuple(rgb_to_i420(np.array(rgb, np.uint8).reshape(1, 1, 3))) == want, rgb


def test_reference_3x3_replicates_the_edge():
    """3x3: chroma is 2x2; samples on the right column and bottom row average the replicated edge pixels."""
    rgb = np.zeros((3, 3, 3), np.uint8)
    rgb[..., 0] = [[0, 40, 200], [80, 120, 10], [255, 3, 77]]  # R; G = B = 0
    out = rgb_to_i420(rgb)
    y = [((66 * int(r) + 128) >> 8) + 16 for r in rgb[..., 0].ravel()]
    assert list(out[:9]) == y
    # R' per sample: (0,0): (0+40+80+120+2)>>2 = 60; (1,0): cols 2,2 -> (200+200+10+10+2)>>2 = 105;
    # (0,1): rows 2,2 -> (255+3+255+3+2)>>2 = 129; (1,1): pixel (2,2) four times -> 77
    means = [60, 105, 129, 77]
    assert list(out[9:13]) == [((-38 * m + 128) >> 8) + 128 for m in means]
    assert list(out[13:17]) == [((112 * m + 128) >> 8) + 128 for m in means]


def test_argument_errors_without_device(built):
    """Null pointers, n <= 0, unknown layouts, bad sizes and short strides are refused, with a message naming the
    problem, before anything touches the engine."""
    from vp8_b200 import _capi
    lib = _capi.load()
    dummy = (C.c_uint8 * 64)()
    p = C.cast(dummy, C.c_void_p)
    arr = (C.c_void_p * 1)(p)
    fake = p  # never dereferenced: the checks below come first
    fb = helpers.i420_bytes(16, 16)

    def key(e=fake, n=1, s=arr, src=p, stride=fb, layout=0, w=16, h=16, q=40, out=arr):
        return lib.vp8r_encode_key_frames_device(e, n, s, src, stride, layout, None, w, h, q, 0, 0, 1, out)

    def inter(stride=fb, layout=0, sr=16):
        return lib.vp8r_encode_inter_frames_device(fake, 1, arr, p, stride, layout, None, 16, 16, 40, 0, 0, sr, arr)

    def conv(e=fake, n=1, src=p, stride=fb, layout=0, w=16, h=16, dst=p, dst_stride=fb):
        return lib.vp8r_convert_to_i420_device(e, n, src, stride, layout, w, h, dst, dst_stride, None)

    cases = [(lambda: key(e=None), "null engine"), (lambda: key(s=None), "null engine"), (lambda: key(src=None), "null engine"),
             (lambda: key(out=None), "null engine"), (lambda: key(n=0), "n <= 0"), (lambda: key(n=-3), "n <= 0"),
             (lambda: key(layout=4), "unknown layout"), (lambda: key(layout=-1), "unknown layout"),
             (lambda: key(w=0), "frame size"), (lambda: key(h=16384), "frame size"), (lambda: key(q=128), "out of range"),
             (lambda: key(stride=fb - 1), "stride smaller"), (lambda: key(layout=2, stride=fb), "stride smaller"),
             (lambda: inter(layout=9), "unknown layout"), (lambda: inter(stride=3), "stride smaller"),
             (lambda: inter(sr=3), "search_range"), (lambda: inter(sr=25), "search_range"),
             (lambda: conv(e=None), "null engine"), (lambda: conv(src=None), "null engine"), (lambda: conv(dst=None), "null engine"),
             (lambda: conv(n=0), "n <= 0"), (lambda: conv(layout=7), "unknown layout"), (lambda: conv(w=-1), "frame size"),
             (lambda: conv(layout=3, stride=fb), "stride smaller"), (lambda: conv(dst_stride=fb - 1), "dst_stride smaller")]
    for k, (call, msg) in enumerate(cases):
        assert call() == VP8R_ERR_INVALID_ARG, k
        assert msg in lib.vp8r_last_error().decode(), (k, lib.vp8r_last_error())


# ---- GPU tier --------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def engine(built):
    import vp8_b200
    e = vp8_b200.Engine(0)
    yield e
    e.close()


def frame_arrays(f):
    """Header, records and coded coefficient blocks of an encoded frame.  Only the coded blocks of a record
    (popcount(coef_mask) from coef_offset) are defined: the rest of the 25 reserved per macroblock is scratch."""
    d = f.desc()
    recs, blocks = [], []
    for m in range(d.hdr.mb_cols * d.hdr.mb_rows):
        r = d.mbs[m]
        recs.append((r.flags, r.coef_mask, r.coef_offset, r.mv[0], r.mv[1], r.aux[0], r.aux[1]))
        nb = bin(r.coef_mask).count("1")
        blocks.append(C.string_at(C.addressof(d.payload.contents) + 32 * r.coef_offset, 32 * nb))
    return bytes(d.hdr), recs, blocks


def scene(n, w, h, frames, seed):
    """n streams of `frames` cropped I420 pictures: a smooth texture under a per-stream pan, with noise."""
    rng = np.random.default_rng(seed)
    m = 2 * frames + 8
    tex = rng.integers(0, 256, (h + 2 * m + 2, w + 2 * m + 2)).astype(np.float32)
    tex = (tex[:-2, :-2] + tex[2:, 2:] + tex[1:-1, 1:-1] * 2 + tex[:-2, 2:] + tex[2:, :-2]) / 6
    cw, ch = (w + 1) // 2, (h + 1) // 2
    out = []
    for s in range(n):
        vy, vx = int(rng.integers(-2, 3)), int(rng.integers(-2, 3))
        pics = []
        for t in range(frames):
            y0, x0 = m + vy * t, m + vx * t
            y = np.clip(tex[y0:y0 + h, x0:x0 + w] + rng.integers(-3, 4, (h, w)), 0, 255).astype(np.uint8)
            u = np.clip(tex[m:m + ch, m + t:m + t + cw] * 0.5 + 64, 0, 255).astype(np.uint8)
            v = np.clip(tex[m + t:m + t + ch, m:m + cw] * 0.5 + 64, 0, 255).astype(np.uint8)
            pics.append(y.tobytes() + u.tobytes() + v.tobytes())
        out.append(pics)
    return out


def assert_same_frames(fa, fb, what):
    for k, (a, b) in enumerate(zip(fa, fb)):
        assert frame_arrays(a) == frame_arrays(b), (what, k)
        assert a.write_bitstream() == b.write_bitstream(), (what, k)


def encode_chain(engine, host_pics, dev_src, w, h, bpred, layout, n_inter=5):
    """Key frame (+ n_inter inter frames) of len(host_pics) streams twice: from the host I420 pictures and from the
    device source dev_src(t) in `layout`; asserts identical records, blocks, bitstreams and reconstructions."""
    n = len(host_pics)
    hs = [engine.open_stream() for _ in range(n)]
    ds = [engine.open_stream() for _ in range(n)]
    try:
        for t in range(1 + n_inter):
            imgs = [host_pics[s][t] for s in range(n)]
            if t == 0:
                fa = engine.encode_key_frames(hs, imgs, w, h, 40, 16, 0, bpred)
                fb = engine.encode_key_frames(ds, dev_src(t), w, h, 40, 16, 0, bpred, layout=layout)
            else:
                fa = engine.encode_inter_frames(hs, imgs, w, h, 40, 16, 0, 8)
                fb = engine.encode_inter_frames(ds, dev_src(t), w, h, 40, 16, 0, 8, layout=layout)
            assert_same_frames(fa, fb, (layout, w, h, t))
            for a, b in zip(hs, ds):
                assert a.read_frame() == b.read_frame(), (layout, w, h, t)
            for f in fa + fb:
                f.close()
    finally:
        for st in hs + ds:
            st.close()


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("size", [(1, 1), (3, 3), (65, 33), (176, 144), (1920, 1080)])
def test_convert_to_i420_matches_numpy(engine, layout, size):
    """Three frames at an odd source address with a stride past the frame, into an odd destination address with a
    stride past the frame; and the tensor API (frames back to back: odd offsets where the frame size is odd)."""
    import torch
    w, h = size
    frames = [source_frame(layout, w, h, 1000 * w + h + k) for k in range(3)]
    want = [img for _, img in frames]
    got = engine.convert_to_i420(torch.from_numpy(np.stack([f for f, _ in frames])).cuda(), layout, w, h)
    assert tuple(got.shape) == (3, helpers.i420_bytes(w, h))
    for k in range(3):
        assert got[k].cpu().numpy().tobytes() == want[k], k
    fb, ob = frames[0][0].size, helpers.i420_bytes(w, h)
    stride, dstride = fb + 37, ob + 5
    src = torch.zeros(1 + 3 * stride, dtype=torch.uint8, device="cuda")
    for k, (f, _) in enumerate(frames):
        src[1 + k * stride:1 + k * stride + fb] = torch.from_numpy(f.reshape(-1)).cuda()
    dst = torch.full((3 + 3 * dstride,), 7, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream or 1
    from vp8_b200.decoder import DEVICE_LAYOUTS
    assert engine._lib.vp8r_convert_to_i420_device(engine.handle, 3, C.c_void_p(src.data_ptr() + 1), stride,
                                                   DEVICE_LAYOUTS[layout], w, h, C.c_void_p(dst.data_ptr() + 3), dstride,
                                                   C.c_void_p(stream)) == 0
    out = dst.cpu().numpy()
    for k in range(3):
        assert out[3 + k * dstride:3 + k * dstride + ob].tobytes() == want[k], k
        assert (out[3 + k * dstride + ob:3 + (k + 1) * dstride] == 7).all()  # nothing written past a frame
    assert (out[:3] == 7).all()


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(176, 144), (65, 33), (320, 240), (1280, 720)])
@pytest.mark.parametrize("bpred", [True, False])
def test_i420_tensor_equals_bytes(engine, size, bpred):
    """Four streams per call: key frame and five inter frames from a CUDA tensor equal the host path."""
    import torch
    w, h = size
    pics = scene(4, w, h, 6, seed=w + h + bpred)
    dev = [torch.from_numpy(np.stack([np.frombuffer(pics[s][t], np.uint8) for s in range(4)])).cuda() for t in range(6)]
    encode_chain(engine, pics, lambda t: dev[t], w, h, bpred, "i420", n_inter=5 if bpred else 0)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["nv12", "rgb", "rgb_planar"])
@pytest.mark.parametrize("size", [(176, 144), (65, 33)])
def test_other_layouts_equal_host_path_of_their_i420(engine, layout, size):
    """NV12 / RGB24 / RGB planar from a CUDA tensor equal the host path fed with convert_to_i420's output."""
    import torch
    w, h = size
    n, steps = 4, 4
    src = [torch.from_numpy(np.stack([source_frame(layout, w, h, 77 * t + s)[0] for s in range(n)])).cuda() for t in range(steps)]
    conv = [engine.convert_to_i420(x, layout, w, h).cpu().numpy() for x in src]
    for t in range(steps):  # and convert_to_i420 is the numpy conversion
        for s in range(n):
            assert conv[t][s].tobytes() == source_frame(layout, w, h, 77 * t + s)[1]
    pics = [[conv[t][s].tobytes() for t in range(steps)] for s in range(n)]
    encode_chain(engine, pics, lambda t: src[t], w, h, True, layout, n_inter=steps - 1)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["i420", "rgb"])
def test_producer_stream_ordering(engine, layout):
    """The input is written on a side stream behind a sleep and the encode is called with that stream current: the
    engine's stream waits for it, and the result equals the host path."""
    import torch
    w, h, n = 176, 144, 4
    frames = [[source_frame(layout, w, h, 500 + 10 * t + s) for s in range(n)] for t in range(3)]
    host = [torch.from_numpy(np.stack([f for f, _ in fr])).pin_memory() for fr in frames]
    side = torch.cuda.Stream()
    hs = [engine.open_stream() for _ in range(n)]
    ds = [engine.open_stream() for _ in range(n)]
    try:
        for t in range(3):
            with torch.cuda.stream(side):
                dev = torch.empty(host[t].shape, dtype=torch.uint8, device="cuda")
                torch.cuda._sleep(50_000_000)  # tens of milliseconds ahead of the copy on the producer stream
                dev.copy_(host[t], non_blocking=True)
                enc = engine.encode_key_frames if t == 0 else engine.encode_inter_frames
                fb = enc(ds, dev, w, h, 40, 16, layout=layout)
            fa = (engine.encode_key_frames if t == 0 else engine.encode_inter_frames)(hs, [img for _, img in frames[t]], w, h, 40, 16)
            assert_same_frames(fa, fb, t)
            for a, b in zip(hs, ds):
                assert a.read_frame() == b.read_frame(), t
            for f in fa + fb:
                f.close()
        side.synchronize()
    finally:
        for st in hs + ds:
            st.close()


@pytest.mark.gpu
def test_transcode_without_pcie(engine):
    """decode_ivf(layout="i420") -> encode_ivf(tensor, layout="i420") gives the IVF bytes of encoding the host
    read-back of the same decode."""
    import vp8_b200
    path = os.path.join(helpers.VEC_DIR, "vp80-02-inter-1402.ivf")
    frames = vp8_b200.decode_ivf(path, engine=engine, layout="i420")[:8]
    imgs = vp8_b200.decode_ivf(path, engine=engine)[:8]
    (_, w, h), = {g for g in helpers.golden_md5(path)[:1]}
    assert tuple(frames.shape) == (8, helpers.i420_bytes(w, h))
    want = vp8_b200.encode_ivf(imgs, w, h, 36, key_interval=5, loop_filter_level=10, engine=engine)
    got = vp8_b200.encode_ivf(frames, w, h, 36, key_interval=5, loop_filter_level=10, engine=engine, layout="i420")
    assert got == want


def _cudart():
    import nvidia.cuda_runtime
    lib = C.CDLL(os.path.join(list(nvidia.cuda_runtime.__path__)[0], "lib", "libcudart.so.12"))
    lib.cudaMallocManaged.argtypes = [C.POINTER(C.c_void_p), C.c_size_t, C.c_uint]
    lib.cudaFree.argtypes = [C.c_void_p]
    return lib


@pytest.mark.gpu
def test_rejections_leave_engine_and_streams_working(engine):
    """Host (pageable), pinned and managed sources and a short stride are refused by the C calls; a tensor on the
    wrong device, non-contiguous or mis-shaped by Python.  After each refusal the same engine and streams encode the
    next inter frame exactly as the host path does."""
    import torch
    w, h, n = 65, 33, 2
    fb = helpers.i420_bytes(w, h)
    pics = scene(n, w, h, 12, seed=9)
    hs = [engine.open_stream() for _ in range(n)]
    ds = [engine.open_stream() for _ in range(n)]
    cudart = _cudart()
    managed = C.c_void_p()
    assert cudart.cudaMallocManaged(C.byref(managed), n * fb, 1) == 0
    pinned = torch.zeros((n, fb), dtype=torch.uint8, pin_memory=True)
    pageable = (C.c_uint8 * (n * fb))()
    good = torch.zeros((n, fb), dtype=torch.uint8, device="cuda")
    lib = engine._lib
    sa = (C.c_void_p * n)(*[s.handle for s in ds])
    step = [0]

    def next_frame(key=False):
        t = step[0]
        step[0] += 1
        imgs = [pics[s][t] for s in range(n)]
        dev = torch.from_numpy(np.stack([np.frombuffer(x, np.uint8) for x in imgs])).cuda()
        if key:
            fa, fb_ = engine.encode_key_frames(hs, imgs, w, h, 40, 8), engine.encode_key_frames(ds, dev, w, h, 40, 8)
        else:
            fa, fb_ = engine.encode_inter_frames(hs, imgs, w, h, 40, 8), engine.encode_inter_frames(ds, dev, w, h, 40, 8)
        assert_same_frames(fa, fb_, t)
        for a, b in zip(hs, ds):
            assert a.read_frame() == b.read_frame(), t

    def c_call(ptr, stride):
        out = [__import__("vp8_b200").ParsedFrame() for _ in range(n)]
        fa = (C.c_void_p * n)(*[f.handle for f in out])
        return lib.vp8r_encode_inter_frames_device(engine.handle, n, sa, C.c_void_p(ptr), stride, 0, None, w, h, 40, 8, 0,
                                                   16, fa)

    try:
        next_frame(key=True)
        for ptr in (C.addressof(pageable), pinned.data_ptr(), managed.value):
            assert c_call(ptr, fb) == VP8R_ERR_INVALID_ARG
            assert "not device memory" in lib.vp8r_last_error().decode()
            next_frame()
        assert c_call(good.data_ptr(), fb - 1) == VP8R_ERR_INVALID_ARG
        assert "stride smaller" in lib.vp8r_last_error().decode()
        next_frame()
        bad = [good.cpu(), torch.zeros((n, 2 * fb), dtype=torch.uint8, device="cuda")[:, ::2], good[:, :fb - 1].contiguous(),
               good[:1], good.view(-1), good.to(torch.int16)]
        for x in bad:
            with pytest.raises(ValueError):
                engine.encode_inter_frames(ds, x, w, h, 40, 8)
            next_frame()
        with pytest.raises(ValueError):
            engine.encode_inter_frames(ds, good, w, h, 40, 8, layout="bgr")
        with pytest.raises(ValueError):
            engine.encode_inter_frames(ds, [pics[0][0]] * n, w, h, 40, 8, layout="rgb")
        next_frame()
    finally:
        cudart.cudaFree(managed)
        for st in hs + ds:
            st.close()
