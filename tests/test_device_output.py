"""Frames delivered into device memory (vp8r_read_batch_device, Engine.read_batch_device, BatchDecoder.decode(out_device=),
decode_ivf(layout=)): I420 / NV12 equal the host read-backs byte for byte, the RGB layouts equal the numpy BT.601
conversion below bit for bit, and the conversion is ordered against a torch consumer on another stream.  The CPU tier
checks the reference conversion itself and the argument checks that need no device."""
import ctypes as C
import os

import numpy as np
import pytest

import helpers

VP8R_ERR_INVALID_ARG, VP8R_ERR_STATE = 1, 5


# ---- reference conversion: BT.601 limited range, chroma point-sampled, integers with an arithmetic shift -------------
def yuv_to_rgb(y, u, v):
    """Arrays of Y, U, V samples (any integer dtype, same shape) -> uint8 array of shape (..., 3)."""
    c, d, e = y.astype(np.int32) - 16, u.astype(np.int32) - 128, v.astype(np.int32) - 128
    r = (298 * c + 409 * e + 128) >> 8
    g = (298 * c - 100 * d - 208 * e + 128) >> 8
    b = (298 * c + 516 * d + 128) >> 8
    return np.clip(np.stack([r, g, b], axis=-1), 0, 255).astype(np.uint8)


def rgb_from_i420(img, w, h, planar=False):
    """Cropped I420 bytes -> (h, w, 3) RGB, or (3, h, w) with `planar`; the chroma sample at (x>>1, y>>1) serves its
    2x2 luma pixels (chroma planes are ceil(w/2) x ceil(h/2))."""
    a = np.frombuffer(img, np.uint8)
    cw, ch = (w + 1) // 2, (h + 1) // 2
    y = a[:w * h].reshape(h, w)
    u = a[w * h:w * h + cw * ch].reshape(ch, cw).repeat(2, 0).repeat(2, 1)[:h, :w]
    v = a[w * h + cw * ch:w * h + 2 * cw * ch].reshape(ch, cw).repeat(2, 0).repeat(2, 1)[:h, :w]
    rgb = yuv_to_rgb(y, u, v)
    return np.ascontiguousarray(rgb.transpose(2, 0, 1)) if planar else rgb


def nv12_from_i420(img, w, h):
    cn = ((w + 1) // 2) * ((h + 1) // 2)
    a = np.frombuffer(img, np.uint8)
    uv = np.stack([a[w * h:w * h + cn], a[w * h + cn:w * h + 2 * cn]], axis=1).reshape(-1)
    return a[:w * h].tobytes() + uv.tobytes()


def layout_bytes(w, h, layout):
    return helpers.i420_bytes(w, h) if layout in ("i420", "nv12") else 3 * w * h


def expected(img, w, h, layout):
    """The bytes a device read-back in `layout` writes for the cropped I420 frame `img`."""
    if layout == "i420":
        return img
    if layout == "nv12":
        return nv12_from_i420(img, w, h)
    return rgb_from_i420(img, w, h, planar=layout == "rgb_planar").tobytes()


# ---- CPU tier --------------------------------------------------------------------------------------------------------
def test_reference_conversion_within_one_of_float_bt601():
    """Every (Y, U, V) triple: the integer conversion is within 1 of the rounded floating-point BT.601 limited-range
    matrix (Kr = 0.299, Kb = 0.114; luma scaled by 255/219, chroma by 255/224)."""
    ky, kc = 255.0 / 219.0, 255.0 / 224.0
    u, v = np.meshgrid(np.arange(256), np.arange(256), indexing="ij")
    u, v = u.reshape(-1), v.reshape(-1)
    d, e = (u - 128) * kc, (v - 128) * kc
    worst = 0
    for yv in range(256):
        y = np.full_like(u, yv)
        got = yuv_to_rgb(y, u, v).astype(np.int32)
        c = (yv - 16) * ky
        ref = np.stack([c + 1.402 * e,
                        c - (1.772 * 0.114 / 0.587) * d - (1.402 * 0.299 / 0.587) * e,
                        c + 1.772 * d], axis=-1)
        ref = np.clip(np.rint(ref), 0, 255).astype(np.int32)
        worst = max(worst, int(np.abs(got - ref).max()))
    assert worst <= 1, worst


def test_reference_conversion_pinned_values():
    pts = {(16, 128, 128): (0, 0, 0),         # black
           (235, 128, 128): (255, 255, 255),  # white
           (126, 128, 128): (128, 128, 128),  # mid grey: (298*110 + 128) >> 8
           (81, 90, 240): (255, 0, 0),        # BT.601 red
           (145, 54, 34): (0, 255, 1),        # BT.601 green: B = (38442 - 38184 + 128) >> 8
           (41, 240, 110): (0, 0, 255),       # BT.601 blue
           (0, 0, 0): (0, 135, 0),            # below the range: G = (-4768 + 12800 + 26624 + 128) >> 8
           (255, 255, 255): (255, 125, 255)}  # above it: G = (71234 - 12700 - 26416 + 128) >> 8
    for (y, u, v), want in pts.items():
        got = tuple(int(x) for x in yuv_to_rgb(np.array([y]), np.array([u]), np.array([v]))[0])
        assert got == want, ((y, u, v), got)


def test_rgb_from_i420_odd_size_point_sampling():
    """3x3 frame: chroma is 2x2, the sample at (x>>1, y>>1) serves each pixel."""
    w = h = 3
    img = bytes([16, 126, 235] * 3) + bytes([128, 240, 128, 54]) + bytes([128, 110, 128, 34])
    rgb = rgb_from_i420(img, w, h)
    assert rgb.shape == (3, 3, 3)
    assert tuple(rgb[0, 0]) == (0, 0, 0) and tuple(rgb[0, 2]) == tuple(yuv_to_rgb(np.array([235]), np.array([240]), np.array([110]))[0])
    assert (rgb_from_i420(img, w, h, planar=True) == rgb.transpose(2, 0, 1)).all()


def test_read_batch_device_argument_errors_without_device(built):
    """Null engine / streams / dst, n <= 0 and an unknown layout are refused before anything touches the engine."""
    from vp8_b200 import _capi
    lib = _capi.load()
    dummy = (C.c_uint8 * 64)()
    sa = (C.c_void_p * 1)(C.cast(dummy, C.c_void_p))
    fake_engine = C.cast(dummy, C.c_void_p)  # never dereferenced: the checks below come first
    assert lib.vp8r_read_batch_device(None, 1, sa, C.cast(dummy, C.c_void_p), 64, 2, None) == VP8R_ERR_INVALID_ARG
    assert lib.vp8r_read_batch_device(fake_engine, 1, None, C.cast(dummy, C.c_void_p), 64, 2, None) == VP8R_ERR_INVALID_ARG
    assert lib.vp8r_read_batch_device(fake_engine, 1, sa, None, 64, 2, None) == VP8R_ERR_INVALID_ARG
    assert lib.vp8r_read_batch_device(fake_engine, 0, sa, C.cast(dummy, C.c_void_p), 64, 2, None) == VP8R_ERR_INVALID_ARG
    for layout in (-1, 4, 99):
        assert lib.vp8r_read_batch_device(fake_engine, 1, sa, C.cast(dummy, C.c_void_p), 64, layout, None) == VP8R_ERR_INVALID_ARG
        assert "unknown layout" in lib.vp8r_last_error().decode()


# ---- GPU tier --------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def engine(built):
    import vp8_b200
    e = vp8_b200.Engine(0)
    yield e
    e.close()


def shown_streams(dec, live, frames):
    """Indices (into dec.streams) of the streams whose frame of this step is shown, in the order the rows are filled."""
    return [i for i, f in zip(live, frames) if f.desc().hdr.show_frame]


@pytest.mark.gpu
def test_all_vectors_device_i420_and_nv12(engine):
    """The 43 vectors as one batch: every shown frame in a device ring in I420 against the golden MD5, and the NV12
    device read-back of each step against the NV12 packed host read-back of the same step."""
    import torch
    import vp8_b200
    vecs = helpers.vectors()
    payloads = [vp8_b200.read_ivf(v)[1] for v in vecs]
    golds = [helpers.golden_md5(v) for v in vecs]
    stride = max(helpers.i420_bytes(w, h) for g in golds for _, w, h in g)
    n = len(vecs)
    dec = vp8_b200.BatchDecoder(engine, n, pinned=True, depth=2)
    ring = [torch.zeros((n, stride), dtype=torch.uint8, device="cuda") for _ in range(2)]
    nv12_dev = torch.zeros((n, stride), dtype=torch.uint8, device="cuda")
    nv12_host = (C.c_uint8 * (n * stride))()
    got = [[] for _ in vecs]

    def on_step(t, live, frames):
        idx = shown_streams(dec, live, frames)
        if not idx:
            return
        rows = ring[t % 2][:len(idx)].cpu().numpy()  # on torch's current stream, behind the conversion
        for k, i in enumerate(idx):
            got[i].append(helpers.md5(rows[k, :dec.streams[i].frame_bytes()].tobytes()))
        sts = [dec.streams[i] for i in idx]
        engine.read_batch_device(sts, nv12_dev, "nv12")
        engine.read_batch_packed(sts, C.addressof(nv12_host), stride, layout="nv12")
        dev = nv12_dev[:len(idx)].cpu().numpy()
        host = np.frombuffer(nv12_host, np.uint8).reshape(n, stride)
        for k, st in enumerate(sts):
            nb = st.frame_bytes()
            assert (dev[k, :nb] == host[k, :nb]).all(), (os.path.basename(vecs[idx[k]]), t)

    dec.decode(payloads, out_device=(ring, "i420"), on_step=on_step)
    dec.close()
    for i, v in enumerate(vecs):
        assert got[i] == [m for m, _, _ in golds[i]], os.path.basename(v)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["rgb", "rgb_planar"])
def test_all_vectors_device_rgb(engine, layout):
    """The 43 vectors as one batch, RGB into a device ring: every shown frame equals the numpy conversion of the same
    frame's I420 (packed host read-back of the step), bit for bit.  Sizes include odd ones and a mid-stream change."""
    import torch
    import vp8_b200
    vecs = helpers.vectors()
    payloads = [vp8_b200.read_ivf(v)[1] for v in vecs]
    golds = [helpers.golden_md5(v) for v in vecs]
    stride = max(3 * w * h for g in golds for _, w, h in g)
    n = len(vecs)
    dec = vp8_b200.BatchDecoder(engine, n, pinned=True, depth=2)
    ring = [torch.zeros((n, stride), dtype=torch.uint8, device="cuda") for _ in range(2)]
    host = (C.c_uint8 * (n * stride))()
    counts = [0] * n

    def on_step(t, live, frames):
        idx = shown_streams(dec, live, frames)
        if not idx:
            return
        sts = [dec.streams[i] for i in idx]
        engine.read_batch_packed(sts, C.addressof(host), stride)
        rows = ring[t % 2][:len(idx)].cpu().numpy()
        yuv = np.frombuffer(host, np.uint8).reshape(n, stride)
        for k, st in enumerate(sts):
            w, h = st.dims()
            want = expected(yuv[k, :st.frame_bytes()].tobytes(), w, h, layout)
            assert rows[k, :3 * w * h].tobytes() == want, (os.path.basename(vecs[idx[k]]), t)
            counts[idx[k]] += 1

    dec.decode(payloads, out_device=(ring, layout), on_step=on_step)
    dec.close()
    assert counts == [len(g) for g in golds]


SYNTH_CASES = ["tiny_odd_intra30", "odd_bilinear_4parts", "qvga_fullpixel_8parts_gop6"]


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["i420", "rgb", "rgb_planar"])
def test_synthetic_mixed_sizes_shown_only(engine, layout):
    """Odd sizes and hidden alt-ref frames, three sizes in one batch with the stride of the largest frame, a packed
    host read-back ring alongside: row k of a step's ring entry is the k-th shown frame of the step."""
    import torch
    import vp8_b200
    m = helpers.synth_manifest()
    ivfs = [helpers.synth_stream(m[name]["args"]) for name in SYNTH_CASES]
    payloads = [vp8_b200.read_ivf(v)[1] for v in ivfs]
    golds = [helpers.synth_golden(name) for name in SYNTH_CASES]
    want = [vp8_b200.decode_ivf(v, engine=engine) for v in ivfs]  # host read-back, checked against the MD5s
    for name, imgs, g in zip(SYNTH_CASES, want, golds):
        assert [helpers.md5(x) for x in imgs] == g, name
    dims = [(int(m[name]["args"].split()[1]), int(m[name]["args"].split()[3])) for name in SYNTH_CASES]
    stride = max(layout_bytes(w, h, layout) for w, h in dims)
    pstride = max(helpers.i420_bytes(w, h) for w, h in dims)
    n, depth = len(SYNTH_CASES), 2
    dec = vp8_b200.BatchDecoder(engine, n, pinned=True, depth=depth)
    ring = [torch.zeros((n, stride), dtype=torch.uint8, device="cuda") for _ in range(depth)]
    packed = [torch.zeros((n, pstride), dtype=torch.uint8, pin_memory=True) for _ in range(depth)]
    got = [[] for _ in range(n)]

    def on_step(t, live, frames):
        engine.sync()  # the packed ring entry of this step has arrived too
        idx = shown_streams(dec, live, frames)
        rows = ring[t % depth][:len(idx)].cpu().numpy()
        for k, i in enumerate(idx):
            w, h = dims[i]
            got[i].append(rows[k, :layout_bytes(w, h, layout)].tobytes())
            assert packed[t % depth][k, :helpers.i420_bytes(w, h)].numpy().tobytes() == want[i][len(got[i]) - 1]

    dec.decode(payloads, out_device=(ring, layout), out_packed=(tuple(p.data_ptr() for p in packed), pstride),
               on_step=on_step)
    dec.close()
    for i, name in enumerate(SYNTH_CASES):
        w, h = dims[i]
        assert got[i] == [expected(img, w, h, layout) for img in want[i]], name


@pytest.mark.gpu
def test_device_parse_1080p_rgb(engine):
    """16 1080p streams with the bitstream parsed on the device: RGB24 rows against numpy of the same step's I420."""
    import torch
    import vp8_b200
    args = "--width 1920 --height 1080 --frames 4 --log2-parts 2 --q 40 --lf 24 --pct-skip 55 --coef-density 3 --pct-empty-block 80"
    n, w, h = 16, 1920, 1080
    payloads = [vp8_b200.read_ivf(helpers.synth_stream(f"{args} --seed {7122 + k}"))[1] for k in range(n)]
    dec = vp8_b200.BatchDecoder(engine, n, pinned=True, device_parse=True, depth=2)
    ring = [torch.empty((n, h, w, 3), dtype=torch.uint8, device="cuda") for _ in range(2)]
    fb = helpers.i420_bytes(w, h)
    host = (C.c_uint8 * (n * fb))()
    steps = []

    def on_step(t, live, frames):
        idx = shown_streams(dec, live, frames)
        engine.read_batch_packed([dec.streams[i] for i in idx], C.addressof(host), fb)
        rows = ring[t % 2][:len(idx)].cpu().numpy()
        yuv = np.frombuffer(host, np.uint8).reshape(n, fb)
        for k in range(len(idx)):
            assert (rows[k] == rgb_from_i420(yuv[k].tobytes(), w, h)).all(), (idx[k], t)
        steps.append(len(idx))

    dec.decode(payloads, out_device=(ring, "rgb"), on_step=on_step)
    dec.close()
    assert sum(steps) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("engine_stream", ["private", "torch"])
def test_consumer_on_another_stream(built, engine_stream):
    """A torch consumer clones each step's ring entry in on_step with no host synchronisation, behind a sleep on its
    stream, so that it falls behind the decoder; depth 2 over 30 steps rewrites ring entries meanwhile.  The engine
    runs on its private stream (the consumer is another stream: both orderings of vp8r_read_batch_device are needed)
    or on the consumer's torch stream.  Every clone must be its step's frames."""
    import torch
    import vp8_b200
    n, w, h, steps = 6, 320, 240, 30
    ivfs = [helpers.synth_stream(f"--width {w} --height {h} --frames {steps} --seed {300 + k} --log2-parts 1 --hidden-altref 0") for k in range(n)]
    payloads = [vp8_b200.read_ivf(v)[1] for v in ivfs]
    consumer = torch.cuda.Stream()
    eng = vp8_b200.Engine(0, cuda_stream=consumer.cuda_stream if engine_stream == "torch" else None)
    try:
        want = [vp8_b200.decode_ivf(v, engine=eng) for v in ivfs]
        assert all(len(x) == steps for x in want)  # every frame shown: row k of step t is stream k's frame t
        dec = vp8_b200.BatchDecoder(eng, n, pinned=True, depth=2)
        ring = [torch.zeros((n, h, w, 3), dtype=torch.uint8, device="cuda") for _ in range(2)]
        clones = []

        def on_step(t, live, frames):
            torch.cuda._sleep(2_000_000)  # about a millisecond of consumer work queued ahead of the clone
            clones.append(ring[t % 2].clone())

        with torch.cuda.stream(consumer):
            dec.decode(payloads, out_device=(ring, "rgb"), on_step=on_step)
        consumer.synchronize()
        dec.close()
        assert len(clones) == steps
        for t, c in enumerate(clones):
            got = c.cpu().numpy()
            for k in range(n):
                assert (got[k] == rgb_from_i420(want[k][t], w, h)).all(), (k, t)
    finally:
        eng.close()


@pytest.mark.gpu
def test_rejections_leave_the_engine_working(engine):
    """Host memory (pinned or pageable), a stride below a frame, a stream without a frame, tensors of the wrong
    dtype / device / shape and a packed read-back whose staging the allocator refuses are refused; the engine reads back
    and decodes correctly afterwards."""
    import torch
    import vp8_b200
    lib = engine._lib
    ivf = helpers.vectors()[0]
    gold = helpers.golden_md5(ivf)
    _, payloads = vp8_b200.read_ivf(ivf)
    st, empty = engine.open_stream(), engine.open_stream()
    try:
        st.decode(payloads[0])
        w, h = st.dims()
        sa = (C.c_void_p * 1)(st.handle)
        fb = 3 * w * h
        pinned = torch.empty((1, fb), dtype=torch.uint8, pin_memory=True)
        pageable = (C.c_uint8 * fb)()
        dev = torch.empty((1, fb), dtype=torch.uint8, device="cuda")
        for ptr in (pinned.data_ptr(), C.addressof(pageable)):
            assert lib.vp8r_read_batch_device(engine.handle, 1, sa, C.c_void_p(ptr), fb, 2, None) == VP8R_ERR_INVALID_ARG
            assert "not device memory" in lib.vp8r_last_error().decode()
        assert lib.vp8r_read_batch_device(engine.handle, 1, sa, C.c_void_p(dev.data_ptr()), fb - 1, 2, None) == VP8R_ERR_INVALID_ARG
        assert lib.vp8r_read_batch_device(engine.handle, 1, sa, C.c_void_p(dev.data_ptr()), fb, 7, None) == VP8R_ERR_INVALID_ARG
        ea = (C.c_void_p * 1)(empty.handle)
        assert lib.vp8r_read_batch_device(engine.handle, 1, ea, C.c_void_p(dev.data_ptr()), fb, 2, None) == VP8R_ERR_STATE
        for bad in (pinned, dev.to(torch.int16), dev.view(-1), dev[:, :fb - 1].contiguous(),
                    torch.empty((0, fb), dtype=torch.uint8, device="cuda"),
                    torch.empty((1, 2 * fb), dtype=torch.uint8, device="cuda")[:, ::2]):
            with pytest.raises(ValueError):
                engine.read_batch_device([st], bad, "rgb")
        with pytest.raises(ValueError):
            engine.read_batch_device([st], dev, "bgr")
        # a stride of 1 TiB asks for 8 TiB of staging, which the allocator refuses at once; the next packed read-back
        # allocates its staging anew and delivers the same bytes
        ib = helpers.i420_bytes(w, h)
        before, after = (C.c_uint8 * ib)(), (C.c_uint8 * ib)()
        assert lib.vp8r_read_batch_packed(engine.handle, 1, sa, C.addressof(before), ib, 0) == 0
        assert lib.vp8r_read_batch_packed(engine.handle, 1, sa, C.addressof(after), 1 << 40, 0) != 0
        assert lib.vp8r_read_batch_packed(engine.handle, 1, sa, C.addressof(after), ib, 0) == 0
        assert bytes(after) == bytes(before)
        assert lib.vp8r_engine_sync(engine.handle) == 0
    finally:
        st.close()
        empty.close()
    # the engine still decodes, and the device read-back delivers every shown frame
    st = engine.open_stream()
    try:
        md5s = []
        out = torch.empty((1, max(helpers.i420_bytes(gw, gh) for _, gw, gh in gold)), dtype=torch.uint8, device="cuda")
        for p in payloads:
            if st.decode(p):
                engine.read_batch_device([st], out, "i420")
                md5s.append(helpers.md5(out[0, :st.frame_bytes()].cpu().numpy().tobytes()))
        assert md5s == [m for m, _, _ in gold]
    finally:
        st.close()


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["i420", "rgb", "rgb_planar"])
def test_decode_ivf_to_tensor(engine, layout):
    import torch
    import vp8_b200
    name = "tiny_odd_intra30"
    ivf = helpers.synth_stream(helpers.synth_manifest()[name]["args"])
    want = vp8_b200.decode_ivf(ivf, engine=engine)
    got = vp8_b200.decode_ivf(ivf, engine=engine, layout=layout)
    w, h = 33, 17
    shape = {"i420": (helpers.i420_bytes(w, h),), "rgb": (h, w, 3), "rgb_planar": (3, h, w)}[layout]
    assert isinstance(got, torch.Tensor) and got.is_cuda and tuple(got.shape) == (len(want),) + shape
    arr = got.cpu().numpy()
    for k, img in enumerate(want):
        assert arr[k].tobytes() == expected(img, w, h, layout), k
    with pytest.raises(ValueError):  # 1425 changes its size mid-stream
        vp8_b200.decode_ivf(os.path.join(helpers.VEC_DIR, "vp80-03-segmentation-1425.ivf"), engine=engine, layout="rgb")
