"""GPU tier: the CUDA path through the C ABI against the golden MD5s and, byte for byte,
against the oracle on the same parsed frames."""
import os

import pytest

import helpers

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine(built):
    import vp8_b200
    e = vp8_b200.Engine(0)
    yield e
    e.close()


@pytest.fixture(scope="module", params=["auto", "swar"])
def engine_forms(request, built):
    """The same tests with the loop filter the engine would pick (scalar form below 128 filtered frames per batch) and
    with the batch form forced (FilterSwarKernel: four pixel lines per register, eight frames per warp): the engine
    reads VP8R_FILTER when it is created."""
    import vp8_b200
    old = os.environ.get("VP8R_FILTER")
    if request.param == "swar":
        os.environ["VP8R_FILTER"] = "swar"
    try:
        e = vp8_b200.Engine(0)
    finally:
        if old is None:
            os.environ.pop("VP8R_FILTER", None)
        else:
            os.environ["VP8R_FILTER"] = old
    yield e
    e.close()


def first_diff(a, b):
    n = min(len(a), len(b))
    for i in range(n):
        if a[i] != b[i]:
            return i
    return n if len(a) != len(b) else -1


@pytest.mark.parametrize("ivf", helpers.vectors(), ids=lambda p: os.path.basename(p)[:-4])
def test_stream_decode_matches_golden_and_oracle(engine, ivf):
    """One stream at a time through vp8r_stream_decode / vp8r_stream_read_frame (src/decode.cc loop)."""
    import vp8_b200
    gold = helpers.golden_md5(ivf)
    _, payloads = vp8_b200.read_ivf(ivf)
    ps, orc = vp8_b200.Parser(), helpers.Oracle()
    st = engine.open_stream()
    shown = 0
    try:
        for k, p in enumerate(payloads):
            fr = ps.parse(p)
            want = orc.decode(fr)
            is_shown = st.decode(p)
            got = st.read_frame()
            assert is_shown == bool(fr.desc().hdr.show_frame)
            d = first_diff(got, want)
            assert d < 0, f"frame {k}: first differing byte {d} (of {len(want)})"
            assert st.checksum() == engine._lib.vp8r_checksum_i420(got, *st.dims())
            if is_shown:
                md5, w, h = gold[shown]
                assert (w, h) == st.dims()
                assert helpers.md5(got) == md5, f"shown frame {shown}"
                shown += 1
            fr.close()
        assert shown == len(gold)
    finally:
        st.close()
        orc.close()


def test_all_vectors_batched(engine_forms):
    """BASELINE config 2: the whole suite as 43 concurrent streams, one batched launch per time step."""
    engine = engine_forms
    import vp8_b200
    vecs = helpers.vectors()
    payloads = [vp8_b200.read_ivf(v)[1] for v in vecs]
    golds = [helpers.golden_md5(v) for v in vecs]
    parsers = [vp8_b200.Parser() for _ in vecs]
    streams = [engine.open_stream() for _ in vecs]
    shown = [0] * len(vecs)
    try:
        for t in range(max(len(p) for p in payloads)):
            live = [i for i in range(len(vecs)) if t < len(payloads[i])]
            frames = [parsers[i].parse(payloads[i][t]) for i in live]
            engine.reconstruct_batch([streams[i] for i in live], frames)
            engine.sync()
            for i, fr in zip(live, frames):
                if fr.desc().hdr.show_frame:
                    md5, w, h = golds[i][shown[i]]
                    assert helpers.md5(streams[i].read_frame()) == md5, f"{os.path.basename(vecs[i])} frame {shown[i]}"
                    shown[i] += 1
                fr.close()
        assert shown == [len(g) for g in golds]
    finally:
        for s in streams:
            s.close()


@pytest.mark.parametrize("name", sorted(helpers.synth_manifest().keys()))
def test_synthetic_streams_match_reference_md5(engine, name):
    """Synthetic streams (bilinear, full-pixel, simple filter, hidden alt-ref, multi-partition,
    1080p) against MD5s produced by the unmodified reference decoder."""
    import vp8_b200
    m = helpers.synth_manifest()[name]
    frames = vp8_b200.decode_ivf(helpers.synth_stream(m["args"]), engine=engine)
    gold = helpers.synth_golden(name)
    assert len(frames) == len(gold)
    for k, (img, md5) in enumerate(zip(frames, gold)):
        assert helpers.md5(img) == md5, f"{name} shown frame {k}"


def test_gop_segments_as_independent_streams(engine):
    """BASELINE config 5 in small: one long-GOP stream cut at its key frames, the segments decoded
    as independent streams of one batch, stitched output == the reference's MD5s of the unsplit
    stream (goldens from the compiled reference decoder)."""
    import vp8_b200
    from vp8_b200 import shard
    args = "--width 640 --height 368 --frames 24 --seed 31 --key-interval 8 --log2-parts 1"
    ivf = helpers.synth_stream(args)
    whole = [helpers.md5(f) for f in helpers.oracle_decode_ivf(ivf)]
    _, payloads = vp8_b200.read_ivf(ivf)
    segs = shard.split_at_key_frames(payloads)
    assert len(segs) == 3
    dec = vp8_b200.BatchDecoder(engine, len(segs), pinned=True)
    got = {g: [] for g in range(len(segs))}

    def on_step(t, live, frames):
        engine.sync()
        for i, fr in zip(live, frames):
            if fr.desc().hdr.show_frame:
                got[i].append(helpers.md5(dec.streams[i].read_frame()))

    dec.decode([s[1] for s in segs], on_step=on_step)
    dec.close()
    assert [m for g in range(len(segs)) for m in got[g]] == whole


def test_native_cli_matches_golden(built, tmp_path):
    """tools/vp8dec.cc (`./decode in.ivf out.yuv` of the reference) on two golden vectors,
    including the one that changes size mid-stream."""
    import subprocess
    for name in ["vp80-02-inter-1418.ivf", "vp80-03-segmentation-1425.ivf", "vp80-05-sharpness-1439.ivf"]:
        ivf = os.path.join(helpers.VEC_DIR, name)
        out = tmp_path / "o.yuv"
        subprocess.check_call([os.path.join(helpers.ROOT, "vp8_b200", "_lib", "vp8dec"), ivf, str(out)])
        data = out.read_bytes()
        pos = 0
        for md5, w, h in helpers.golden_md5(ivf):
            n = helpers.i420_bytes(w, h)
            assert helpers.md5(data[pos:pos + n]) == md5
            pos += n
        assert pos == len(data)


@pytest.mark.parametrize("host_parse", [False, True], ids=["device-parse", "host-parse"])
def test_native_cli_batch_mode_matches_golden(built, tmp_path, host_parse):
    """vp8dec --batch: the lock-step loop of INTEGRATION.md written in C++ on the C ABI (frame headers on host threads,
    everything else of the parse on the GPU unless --host-parse, packed read-back ring, fences).  Twelve vectors of
    different lengths and sizes as twelve streams, one of them changing its size mid-stream; every shown frame against
    the golden MD5."""
    import subprocess
    names = sorted(os.path.basename(v) for v in helpers.vectors())[:11] + ["vp80-05-sharpness-1439.ivf"]
    names = list(dict.fromkeys(names))
    out_dir = tmp_path / "out"
    out_dir.mkdir()
    cmd = [os.path.join(helpers.ROOT, "vp8_b200", "_lib", "vp8dec")] + (["--host-parse"] if host_parse else []) + \
          ["--batch", str(out_dir)] + [os.path.join(helpers.VEC_DIR, n) for n in names]
    subprocess.check_call(cmd)
    for name in names:
        data = (out_dir / (name + ".yuv")).read_bytes()
        pos = 0
        for md5, w, h in helpers.golden_md5(os.path.join(helpers.VEC_DIR, name)):
            n = helpers.i420_bytes(w, h)
            assert helpers.md5(data[pos:pos + n]) == md5, name
            pos += n
        assert pos == len(data), name


def test_device_resident_replay_and_checksums(engine):
    """vp8r_frame_upload + vp8r_reconstruct_batch on resident frames gives the same pictures as the
    staged path, and the device checksum equals the host checksum of the copied-back frame."""
    import vp8_b200
    ivf = helpers.synth_stream("--width 320 --height 240 --frames 8 --seed 41 --log2-parts 2")
    _, payloads = vp8_b200.read_ivf(ivf)
    ps = vp8_b200.Parser()
    frames = [ps.parse(p) for p in payloads]
    for f in frames:
        engine.upload(f)
    st = engine.open_stream()
    want = helpers.oracle_decode_ivf(ivf)
    k = 0
    for rep in range(2):  # replaying from the key frame must be repeatable
        k = 0
        for f in frames:
            engine.reconstruct_batch([st], [f])
            if f.desc().hdr.show_frame:
                img = st.read_frame()
                assert img == want[k]
                assert st.checksum() == engine._lib.vp8r_checksum_i420(img, *st.dims())
                k += 1
    assert k == len(want)
    st.close()
    for f in frames:
        f.close()


def test_4k_frames_match_oracle_checksums(engine_forms):
    """BASELINE config 5 frame size (3840x2160, 240x135 macroblocks, 8 DCT partitions): every frame's
    device-side checksum equals the checksum of the oracle's picture, and the last frame is compared
    byte for byte."""
    engine = engine_forms
    import vp8_b200
    ivf = helpers.synth_stream("--width 3840 --height 2160 --frames 4 --seed 51 --log2-parts 3 "
                               "--pct-skip 55 --coef-density 3 --pct-empty-block 80 --altref-period 3")
    _, payloads = vp8_b200.read_ivf(ivf)
    ps, orc, st = vp8_b200.Parser(), helpers.Oracle(), engine.open_stream()
    lib = engine._lib
    try:
        for k, p in enumerate(payloads):
            fr = ps.parse(p)
            want = orc.decode(fr)
            st.decode(p)
            assert st.dims() == (3840, 2160)
            assert st.checksum() == lib.vp8r_checksum_i420(want, 3840, 2160), f"frame {k}"
            if k == len(payloads) - 1:
                assert st.read_frame() == want
            fr.close()
    finally:
        st.close()
        orc.close()


def test_many_streams_lockstep_checksums(engine_forms):
    """48 independent streams of different seeds and two sizes in one lock-step batch (the bench's
    execution pattern, band-major filter tickets included): every stream's every frame matches the
    oracle by checksum."""
    engine = engine_forms
    import vp8_b200
    n = 48
    ivfs = [helpers.synth_stream(f"--width {320 if k % 2 else 400} --height {240 if k % 2 else 304} --frames 5 "
                                 f"--seed {100 + k} --log2-parts {k % 3}") for k in range(n)]
    payloads = [vp8_b200.read_ivf(v)[1] for v in ivfs]
    want = []
    for k in range(n):
        ps, orc = vp8_b200.Parser(), helpers.Oracle()
        sums = []
        for p in payloads[k]:
            fr = ps.parse(p)
            img = orc.decode(fr)
            d = fr.desc().hdr
            sums.append(engine._lib.vp8r_checksum_i420(img, d.width, d.height))
            fr.close()
        orc.close()
        want.append(sums)
    dec = vp8_b200.BatchDecoder(engine, n, pinned=True)
    got = [[] for _ in range(n)]

    def on_step(t, live, frames):
        sums = engine.checksum_batch([dec.streams[i] for i in live])
        for i, s in zip(live, sums):
            got[i].append(s)

    dec.decode(payloads, on_step=on_step)
    dec.close()
    assert got == want


@pytest.fixture(scope="module")
def path_engines(built):
    e = helpers.Engines()
    yield e
    e.close()


@pytest.fixture(scope="module")
def randomised_streams(built):
    """The streams of helpers.randomised_configs() and the oracle's checksum of each of their frames."""
    import vp8_b200
    cfgs = helpers.randomised_configs()
    from vp8_b200 import _capi
    payloads = [vp8_b200.read_ivf(helpers.synth_stream(c))[1] for c in cfgs]
    return cfgs, payloads, [helpers.oracle_checksums(_capi.load(), p) for p in payloads]


DEVICE_PATHS = [k for k, v in helpers.DECODE_PATHS.items() if v.get("tokens_on_device") or v.get("device_parse")]


@pytest.mark.parametrize("path", list(helpers.DECODE_PATHS) + [p + "-by-parts" for p in DEVICE_PATHS])
def test_randomised_streams_against_oracle(path_engines, randomised_streams, path):
    """100 small streams with randomised generator settings (helpers.randomised_configs: all four bitstream versions,
    both loop filters, every sharpness, 1-8 partitions, odd sizes, dense SPLIT / intra / B_PRED mixes, GOP lengths,
    DCT_CAT6 magnitudes, vectors far beyond the frame, probability updates, no skip flag, 1 to 25 macroblock rows)
    decoded as one lock-step batch on each decode path; every frame of every stream must equal the oracle's picture
    (device checksum against the checksum of the oracle's output).  The token kernel's instance follows the largest
    partition count of the batch, so the "-by-parts" rows decode the set again as four batches of one partition
    count each."""
    cfgs, payloads, want = randomised_streams
    by_parts = path.endswith("-by-parts")
    row = helpers.DECODE_PATHS[path[:-len("-by-parts")] if by_parts else path]
    engine = path_engines.get(row["env"])
    groups = [list(range(len(cfgs)))]
    if by_parts:
        groups = [[i for i, c in enumerate(cfgs) if f"--log2-parts {lp} " in c] for lp in range(4)]
        assert sorted(i for g in groups for i in g) == list(range(len(cfgs)))
    bad = []
    for g in groups:
        bad += helpers.decode_on_path(engine, [payloads[i] for i in g], [want[i] for i in g], row, [cfgs[i] for i in g])
    assert not bad, f"{len(bad)} frames differ: {bad[:4]}"


def test_packed_readback_equals_pitched_readback(engine_forms):
    """vp8r_read_batch_packed (device-side crop + I420 pack, one copy) against vp8r_stream_read_frame
    for even, odd and tiny frame sizes in one batch."""
    engine = engine_forms
    import ctypes as C
    import vp8_b200
    sizes = [(176, 144), (175, 143), (33, 17), (16, 16), (130, 98), (320, 240)]
    ivfs = [helpers.synth_stream(f"--width {w} --height {h} --frames 3 --seed {70 + k}") for k, (w, h) in enumerate(sizes)]
    streams = [engine.open_stream() for _ in sizes]
    try:
        for st, ivf in zip(streams, ivfs):
            for p in vp8_b200.read_ivf(ivf)[1]:
                st.decode(p)
        stride = max(st.frame_bytes() for st in streams) + 5  # deliberately unaligned stride
        buf = (C.c_uint8 * (stride * len(streams)))()
        engine.read_batch_packed(streams, C.addressof(buf), stride)
        raw = bytes(buf)
        for k, st in enumerate(streams):
            want = st.read_frame()
            assert raw[k * stride:k * stride + len(want)] == want, sizes[k]
        # the NV12 option: same Y plane, then U and V samples interleaved
        engine.read_batch_packed(streams, C.addressof(buf), stride, layout="nv12")
        raw = bytes(buf)
        for k, st in enumerate(streams):
            want = st.read_frame()
            w, h = st.dims()
            cn = ((w + 1) // 2) * ((h + 1) // 2)
            u, v = want[w * h:w * h + cn], want[w * h + cn:]
            nv12 = want[:w * h] + bytes(b for pair in zip(u, v) for b in pair)
            assert raw[k * stride:k * stride + len(want)] == nv12, sizes[k]
    finally:
        for st in streams:
            st.close()


# ---- device-side token decode (deferred tokens, SURVEY 8 row f1) ----------------------------------
def _decode_deferred(engine, payloads, modes=False):
    """All frames of one stream with the DCT partitions (and, with `modes`, the macroblock headers of
    the first partition) decoded on the device; returns the I420 of every frame (shown or not) and
    the show flags."""
    import vp8_b200
    ps = vp8_b200.Parser()
    ps.set_defer_tokens(True)
    if modes:
        ps.set_defer_modes(True)
    st = engine.open_stream()
    out, shown = [], []
    try:
        for p in payloads:
            fr = ps.parse(p, pinned=True)
            assert fr.desc().hdr.tokens_deferred == 1 and fr.desc().hdr.modes_deferred == int(modes)
            engine.reconstruct_batch([st], [fr])
            engine.sync()
            out.append(st.read_frame())
            shown.append(bool(fr.desc().hdr.show_frame))
            fr.close()
    finally:
        st.close()
        ps.close()
    return out, shown


@pytest.mark.parametrize("modes", [False, True], ids=["tokens", "modes+tokens"])
@pytest.mark.parametrize("ivf", helpers.vectors(), ids=lambda p: os.path.basename(p)[:-4])
def test_device_tokens_match_golden_and_oracle(engine, ivf, modes):
    """Host parses the first partition only (or, with `modes`, just the frame header); the parse kernel
    decodes the rest.  Every frame byte for byte against host parser -> oracle, shown frames against
    the golden MD5s."""
    import vp8_b200
    gold = helpers.golden_md5(ivf)
    _, payloads = vp8_b200.read_ivf(ivf)
    got, shown = _decode_deferred(engine, payloads, modes)
    ps, orc = vp8_b200.Parser(), helpers.Oracle()
    k_shown = 0
    for k, p in enumerate(payloads):
        fr = ps.parse(p)
        want = orc.decode(fr)
        fr.close()
        d = first_diff(got[k], want)
        assert d < 0, f"frame {k}: first differing byte {d} (of {len(want)})"
        if shown[k]:
            assert helpers.md5(got[k]) == gold[k_shown][0]
            k_shown += 1
    assert k_shown == len(gold)
    orc.close()


@pytest.mark.parametrize("modes", [False, True], ids=["tokens", "modes+tokens"])
@pytest.mark.parametrize("name", sorted(helpers.synth_manifest().keys()))
def test_device_tokens_synthetic_streams(engine, name, modes):
    """Same, on the synthetic streams (1/2/4/8 DCT partitions, segment quantisers, 1080p)."""
    import vp8_b200
    m = helpers.synth_manifest()[name]
    _, payloads = vp8_b200.read_ivf(helpers.synth_stream(m["args"]))
    got, shown = _decode_deferred(engine, payloads, modes)
    gold = helpers.synth_golden(name)
    imgs = [g for g, s in zip(got, shown) if s]
    assert len(imgs) == len(gold)
    for k, (img, md5) in enumerate(zip(imgs, gold)):
        assert helpers.md5(img) == md5, f"{name} shown frame {k}"


def test_device_tokens_batched_and_truncated(engine):
    """Batched lock-step decode with device tokens == host tokens (device checksums), and an
    over-read DCT partition is reported by vp8r_engine_sync as VP8R_ERR_TRUNCATED."""
    import vp8_b200
    from vp8_b200._capi import Vp8rError
    ivfs = [helpers.synth_stream(f"--width 320 --height 192 --frames 5 --seed {70 + k} --log2-parts {k % 4}") for k in range(6)]
    payloads = [vp8_b200.read_ivf(d)[1] for d in ivfs]
    sums = []
    for tok, par in ((False, False), (True, False), (False, True)):
        dec = vp8_b200.BatchDecoder(engine, len(ivfs), pinned=True, tokens_on_device=tok, device_parse=par)
        per_step = []
        dec.decode(payloads, on_step=lambda t, live, frames: per_step.append(engine.checksum_batch([dec.streams[i] for i in live])))
        sums.append(per_step)
        dec.close()
    assert sums[0] == sums[1] == sums[2]
    # cut the tail of the last partition of a frame with many tokens: the token kernel must flag it
    ps = vp8_b200.Parser()
    ps.set_defer_tokens(True)
    st = engine.open_stream()
    key = payloads[0][0]
    first_size = (key[0] | key[1] << 8 | key[2] << 16) >> 5
    keep = 10 + first_size + (len(key) - 10 - first_size) // 3
    fr = ps.parse(key[:keep], pinned=True)
    engine.reconstruct_batch([st], [fr])
    with pytest.raises(Vp8rError) as ei:
        engine.sync()
    assert ei.value.code == 4
    engine.sync()  # the flag is cleared once reported
    fr.close()
    st.close()


def test_passes_without_draining_and_resident_replays(engine):
    """decode(drain=False) hands the pipeline over to the next pass (new streams after reset, same ring): the frames
    that arrive in the pinned ring are those of a drained pass.  And frames kept resident with a deferred parse
    (their records are rewritten by the parse kernels at every reconstruction) may be replayed back to back."""
    import ctypes as C
    import vp8_b200
    n, depth = 5, 3
    ivfs = [helpers.synth_stream(f"--width 320 --height 192 --frames 7 --seed {270 + k} --log2-parts {k % 3}") for k in range(n)]
    payloads = [vp8_b200.read_ivf(d)[1] for d in ivfs]
    fb = 320 * 192 * 3 // 2
    want = []
    for p in payloads:
        ps, orc = vp8_b200.Parser(), helpers.Oracle()
        imgs = []
        for x in p:
            fr = ps.parse(x)
            img = orc.decode(fr)
            if fr.desc().hdr.show_frame:
                imgs.append(img)
            fr.close()
        orc.close()
        want.append(imgs)
    bufs = [(C.c_uint8 * (n * fb))() for _ in range(depth)]
    packed = (tuple(C.addressof(b) for b in bufs), fb)
    dec = vp8_b200.BatchDecoder(engine, n, pinned=True, device_parse=True, depth=depth)
    got = [[] for _ in range(n)]
    pending = []

    def on_step(t, live, frames):
        # the ring entry of global step g is g % depth; it is complete once its ticket has been waited for
        g = dec._g + t
        pending.append((g, dec._tickets[g], [i for i, f in zip(live, frames) if f.desc().hdr.show_frame]))
        while len(pending) >= depth:
            g0, ticket, shown = pending.pop(0)
            dec.wait(ticket)
            for k, i in enumerate(shown):
                got[i].append(bytes(bufs[g0 % depth][k * fb:(k + 1) * fb]))

    for k in range(3):
        dec.reset()
        dec.decode(payloads, out_packed=packed, on_step=on_step, drain=k == 2)
    for g0, ticket, shown in pending:
        for k, i in enumerate(shown):
            got[i].append(bytes(bufs[g0 % depth][k * fb:(k + 1) * fb]))
    for i in range(n):
        assert got[i] == want[i] * 3, f"stream {i}"
    final_sums = engine.checksum_batch(dec.streams)
    dec.close()
    # resident replays: parse once with deferred modes, upload, reconstruct the same frames pass after pass
    dec = vp8_b200.BatchDecoder(engine, n, pinned=False, device_parse=True)
    resident = []
    for t in range(7):
        frames = dec.parse_into([vp8_b200.ParsedFrame(pinned=False) for _ in range(n)], [p[t] for p in payloads], list(range(n)))
        for f in frames:
            engine.upload(f, release_host=True)
        resident.append(frames)
    sums = []
    for _ in range(4):
        for t in range(7):
            engine.reconstruct_batch(dec.streams, resident[t])
        sums.append(engine.checksum_batch(dec.streams))
    assert sums[0] == sums[1] == sums[2] == sums[3] == final_sums
    for fr in resident:
        for f in fr:
            f.close()
    dec.close()


def _truncated_key_frame():
    """A 320x192 key frame whose declared first partition is cut to half: the start code and headers are kept, the
    macroblock headers then run past the partition's end while the DCT partition (the bytes behind it) is present."""
    import vp8_b200
    ivf = helpers.synth_stream("--width 320 --height 192 --frames 2 --seed 9 --log2-parts 0")
    key = vp8_b200.read_ivf(ivf)[1][0]
    first_size = (key[0] | key[1] << 8 | key[2] << 16) >> 5
    cut = first_size // 2
    tag = (key[0] | key[1] << 8 | key[2] << 16) & 0x1f | (cut << 5)
    return bytes([tag & 0xff, (tag >> 8) & 0xff, (tag >> 16) & 0xff]) + key[3:10 + cut] + key[10 + first_size:]


def test_device_parse_truncated_first_partition(engine):
    """Deferred modes: a first partition that ends early is reported by vp8r_engine_sync
    (VP8R_ERR_TRUNCATED), like the host parser does for the same bytes."""
    import vp8_b200
    from vp8_b200._capi import Vp8rError
    bad = _truncated_key_frame()
    host = vp8_b200.Parser()
    with pytest.raises(Vp8rError) as e0:
        host.parse(bad)
    assert e0.value.code == 4
    ps = vp8_b200.Parser()
    ps.set_defer_modes(True)
    st = engine.open_stream()
    fr = ps.parse(bad, pinned=True)
    engine.reconstruct_batch([st], [fr])
    with pytest.raises(Vp8rError) as e1:
        engine.sync()
    assert e1.value.code == 4
    engine.sync()
    fr.close()
    st.close()


def test_device_parse_failure_survives_encoder_calls(engine):
    """A device-parse failure not yet reported is still reported by vp8r_engine_sync after encoder calls have reused
    the slot of its batch (the encoders harvest the slot's error words as decoded batches do)."""
    import vp8_b200
    from vp8_b200._capi import Vp8rError
    ps = vp8_b200.Parser()
    ps.set_defer_modes(True)
    st, enc = engine.open_stream(), engine.open_stream()
    fr = ps.parse(_truncated_key_frame(), pinned=True)
    engine.reconstruct_batch([st], [fr])
    w, h = 64, 48
    image = bytes(range(256)) * ((w * h * 3 // 2) // 256)
    for _ in range(16):  # more calls than the engine has slots
        for f in engine.encode_key_frames([enc], [image], w, h, q_index=40):
            f.close()
    with pytest.raises(Vp8rError) as e:
        engine.sync()
    assert e.value.code == 4
    engine.sync()
    fr.close()
    st.close()
    enc.close()

def test_device_parse_survives_corrupted_streams(engine):
    """Bit flips / garbage in the partitions (the frame header kept valid): the device-side parse must
    neither hang nor fault; whatever it decodes equals what the host parser + oracle make of the same
    bytes whenever the host parser accepts them."""
    import random
    import vp8_b200
    from vp8_b200._capi import Vp8rError
    rng = random.Random(4242)
    base = helpers.synth_stream("--width 96 --height 80 --frames 5 --seed 5 --log2-parts 2 --pct-split 30 --pct-intra 20")
    _, payloads = vp8_b200.read_ivf(base)
    compared = flagged = 0
    for trial in range(40):
        host, dev, orc = vp8_b200.Parser(), vp8_b200.Parser(), helpers.Oracle()
        dev.set_defer_modes(True)
        st = engine.open_stream()
        try:
            for k, pl in enumerate(payloads):
                data = bytearray(pl)
                hdr = 10 if k == 0 else 3
                lo = hdr + 60  # keep the frame header (probability updates etc.) intact
                for _ in range(rng.randint(1, 6)):
                    data[rng.randrange(lo, len(data))] ^= 1 << rng.randrange(8)
                data = bytes(data)
                host_ok = True
                try:
                    want = orc.decode(host.parse(data))
                except Vp8rError:
                    host_ok = False
                try:
                    fr = dev.parse(data, pinned=True)
                except Vp8rError:
                    break  # header-level rejection: same code path as the host parser
                engine.reconstruct_batch([st], [fr])
                try:
                    engine.sync()
                    dev_ok = True
                except Vp8rError as e:
                    assert e.code == 4
                    dev_ok = False
                    flagged += 1
                fr.close()
                if not (host_ok and dev_ok):
                    break  # the stream is dead for both from here on
                assert st.read_frame() == want, f"trial {trial} frame {k}"
                compared += 1
        finally:
            st.close()
            orc.close()
    assert compared > 40


def test_device_parse_4k_segments(engine):
    """BASELINE config 5 with the device-side parse: a 3840x2160 long-GOP stream cut at its key frames,
    the segments decoded as independent streams of one batch with macroblock headers and tokens decoded
    on the GPU; every frame's device checksum equals the host-parsed decode of the unsplit stream."""
    import vp8_b200
    from vp8_b200 import shard
    ivf = helpers.synth_stream("--width 3840 --height 2160 --frames 8 --seed 77 --key-interval 4 --log2-parts 3 --pct-skip 60")
    _, payloads = vp8_b200.read_ivf(ivf)
    # reference pass: host parse, one stream
    want = []
    ps, st = vp8_b200.Parser(), engine.open_stream()
    for p in payloads:
        fr = ps.parse(p, pinned=True)
        engine.reconstruct_batch([st], [fr])
        engine.sync()
        want.append(st.checksum())
        fr.close()
    st.close()
    segs = shard.split_at_key_frames(payloads)
    assert len(segs) == 2
    dec = vp8_b200.BatchDecoder(engine, len(segs), pinned=True, device_parse=True, depth=3)
    got = {g: [] for g in range(len(segs))}

    def on_step(t, live, frames):
        sums = engine.checksum_batch([dec.streams[i] for i in live])
        for i, s in zip(live, sums):
            got[i].append(s)

    dec.decode([s[1] for s in segs], on_step=on_step)
    dec.close()
    stitched = [c for g in range(len(segs)) for c in got[g]]
    assert stitched == want


@pytest.mark.parametrize("modes", [False, True], ids=["tokens", "modes+tokens"])
def test_device_parse_failure_names_and_stops_the_stream(engine, modes):
    """A frame whose device-side parse runs past a partition is not reconstructed; the error (at the next sync)
    names the stream of the batch; that stream rejects inter frames until its next key frame, the other stream of
    the batch decodes on and stays bit-exact."""
    import vp8_b200
    from vp8_b200._capi import Vp8rError
    good = vp8_b200.read_ivf(helpers.synth_stream("--width 320 --height 192 --frames 8 --seed 21 --log2-parts 1"))[1]
    vict = vp8_b200.read_ivf(helpers.synth_stream("--width 320 --height 192 --frames 8 --seed 22 --log2-parts 1 --key-interval 4"))[1]
    f = vict[2]
    first_size = (f[0] | f[1] << 8 | f[2] << 16) >> 5
    if modes:   # shorten the declared first partition: the macroblock headers run past its end
        cut = first_size // 2
        tag = (f[0] | f[1] << 8 | f[2] << 16) & 0x1f | (cut << 5)
        bad = bytes([tag & 0xff, (tag >> 8) & 0xff, (tag >> 16) & 0xff]) + f[3:3 + cut] + f[3 + first_size:]
    else:       # drop most of the last DCT partition: its token reader runs past the end
        bad = f[:len(f) - (len(f) - 3 - first_size) // 3]
    vict = vict[:2] + [bad] + vict[3:]

    def parser():
        p = vp8_b200.Parser()
        (p.set_defer_modes if modes else p.set_defer_tokens)(True)
        return p

    pg, pv, host, orc = parser(), parser(), vp8_b200.Parser(), helpers.Oracle()
    sg, sv = engine.open_stream(), engine.open_stream()
    try:
        reported = False
        for t in range(8):
            want = orc.decode(host.parse(good[t]))
            fg = pg.parse(good[t], pinned=True)
            if t == 3 and reported:
                # the victim is stopped: its inter frame is refused, the good stream goes on alone
                with pytest.raises(Vp8rError) as e2:
                    engine.reconstruct_batch([sg, sv], [fg, pv.parse(vict[t], pinned=True)])
                assert e2.value.code in (4, 5)
                engine.reconstruct_batch([sg], [fg])
            elif t < 3 or t >= 4:
                try:
                    fv = pv.parse(vict[t], pinned=True)
                except Vp8rError:
                    fv = None  # the host part of the parse may already reject the damaged frame
                if fv is None:
                    engine.reconstruct_batch([sg], [fg])
                else:
                    engine.reconstruct_batch([sg, sv], [fg, fv])
            try:
                engine.sync()
            except Vp8rError as e1:
                assert t == 2 and e1.code == 4 and "stream 1 of the batch" in str(e1)
                reported = True
            assert sg.read_frame() == want, f"good stream, frame {t}"
        assert reported
        # from its key frame (frame 4) on the victim decodes again
        assert sv.frame_bytes() > 0
    finally:
        sg.close()
        sv.close()
        orc.close()
