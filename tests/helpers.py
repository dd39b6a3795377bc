"""Test-side helpers: golden MD5 lists, the oracle binding (oracle/ is test infrastructure and is
only ever loaded from here, from __graft_entry__.smoke() and from bench.py's CPU legs)."""
import ctypes as C
import glob
import hashlib
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VEC_DIR = os.path.join(ROOT, "tests", "golden", "vp8-test-vectors")
SYN_DIR = os.path.join(ROOT, "tests", "golden", "synthetic")
ORACLE_SO = os.path.join(ROOT, "oracle", "_build", "liboracle.so")
LIB_SO = os.path.join(ROOT, "vp8_b200", "_lib", "libvp8r.so")
REF_DECODE = os.path.join(ROOT, "oracle", "_ref", "decode")


def ensure_built():
    if not (os.path.exists(LIB_SO) and os.path.exists(ORACLE_SO)):
        subprocess.check_call([os.path.join(ROOT, "build.sh")], cwd=ROOT)


def vectors():
    """The 43 shipped test vectors, plus every *.ivf with a *.ivf.md5 beside it under $VP8_TEST_VECTORS (the 18
    vp80-00-comprehensive-* vectors are git-ignored in the reference, test/test_comprehensive.py:13-20: supply
    them there and every vector test picks them up)."""
    found = sorted(glob.glob(os.path.join(VEC_DIR, "*.ivf")))
    extra = os.environ.get("VP8_TEST_VECTORS")
    if extra and os.path.isdir(extra):
        have = {os.path.basename(p) for p in found}
        for p in sorted(glob.glob(os.path.join(extra, "**", "*.ivf"), recursive=True)):
            if os.path.exists(p + ".md5") and os.path.basename(p) not in have:
                found.append(p)
    return found


def golden_md5(ivf_path):
    """[(md5, width, height)] per shown frame; the size comes from the md5 line's file name
    (streams 1425 and 1436 change size mid-stream)."""
    out = []
    for line in open(ivf_path + ".md5"):
        md5, name = line.split()
        m = re.search(r"-(\d+)x(\d+)-(\d+)\.i420$", name)
        out.append((md5, int(m.group(1)), int(m.group(2))))
    return out


def i420_bytes(w, h):
    return w * h + 2 * ((w + 1) // 2) * ((h + 1) // 2)


def md5(b):
    return hashlib.md5(b).hexdigest()


class Oracle:
    """ctypes view of oracle/_build/liboracle.so (CPU restatement of the reconstruction path)."""

    def __init__(self):
        ensure_built()
        self.lib = C.CDLL(ORACLE_SO)
        self.lib.oracle_create.restype = C.c_void_p
        self.lib.oracle_destroy.argtypes = [C.c_void_p]
        self.lib.oracle_decode_frame.argtypes = [C.c_void_p, C.c_void_p]
        self.lib.oracle_decode_frame.restype = C.c_int
        self.lib.oracle_frame_bytes.argtypes = [C.c_void_p]
        self.lib.oracle_frame_bytes.restype = C.c_size_t
        self.lib.oracle_write_i420.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        self.lib.oracle_write_i420.restype = C.c_size_t
        self.lib.oracle_idct4x4.argtypes = [C.POINTER(C.c_int16)]
        self.lib.oracle_iwht4x4.argtypes = [C.POINTER(C.c_int16)]
        self.h = self.lib.oracle_create()

    def decode(self, parsed_frame):
        """parsed_frame: vp8_b200.ParsedFrame.  Returns the I420 bytes of the reconstructed frame."""
        d = parsed_frame.desc()
        rc = self.lib.oracle_decode_frame(self.h, C.byref(d))
        if rc != 0:
            raise RuntimeError(f"oracle_decode_frame: {rc}")
        n = self.lib.oracle_frame_bytes(self.h)
        buf = (C.c_uint8 * n)()
        self.lib.oracle_write_i420(self.h, buf, n)
        return bytes(buf)

    def close(self):
        if self.h:
            self.lib.oracle_destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()


def oracle_decode_ivf(path_or_bytes):
    """Shown frames of a stream through host parser -> oracle."""
    import vp8_b200
    _, payloads = vp8_b200.read_ivf(path_or_bytes)
    ps, orc = vp8_b200.Parser(), Oracle()
    out = []
    for p in payloads:
        fr = ps.parse(p)
        img = orc.decode(fr)
        if fr.desc().hdr.show_frame:
            out.append(img)
        fr.close()
    orc.close()
    return out


def ref_decode_ivf(path):
    """The compiled, unmodified reference decoder (oracle/_ref/decode) on a file; raw YUV bytes."""
    import tempfile
    with tempfile.NamedTemporaryFile(suffix=".yuv") as t:
        subprocess.check_call([REF_DECODE, path, t.name])
        return open(t.name, "rb").read()


SYNTH_BIN = os.path.join(ROOT, "vp8_b200", "_lib", "vp8synth")


def synth_manifest():
    import json
    return json.load(open(os.path.join(SYN_DIR, "manifest.json")))


def synth_stream(args):
    """Runs vp8synth with `args` (str) and returns the IVF bytes."""
    import tempfile
    ensure_built()
    with tempfile.TemporaryDirectory() as td:
        p = os.path.join(td, "s.ivf")
        subprocess.check_call([SYNTH_BIN] + args.split() + ["--out", p])
        return open(p, "rb").read()


def synth_golden(name):
    return [l.split()[0] for l in open(os.path.join(SYN_DIR, name + ".md5"))]


# ---- randomised generator settings and the decode paths they run on ----------------------------------------------
def randomised_configs():
    """vp8synth settings of the randomised parity matrix.  The first 60 draws are the original matrix (all four
    versions, both filters, every sharpness, 1-8 partitions, odd sizes, SPLIT / intra / B_PRED mixes, GOP lengths);
    the 40 after them add the syntax extremes (DCT_CAT6 magnitudes, vectors beyond the frame, probability updates,
    no skip flag) and frames of 1, 12, 13, 24 and 25 macroblock rows, across the 12-row bands of the loop filter.
    The 1-row frames use 8 partitions, so some partitions own no row."""
    import random
    rng = random.Random(20261018)
    cfgs = []
    for k in range(60):
        w, h = rng.choice([(16, 16), (17, 33), (48, 64), (96, 80), (130, 98), (176, 144), (250, 120), (320, 16)])
        cfgs.append(f"--width {w} --height {h} --frames {rng.randint(3, 9)} --seed {1000 + k} "
                    f"--version {rng.randint(0, 3)} --filter-type {rng.randint(0, 1)} --sharpness {rng.randint(0, 7)} "
                    f"--lf {rng.choice([0, 1, 8, 24, 40, 63])} --q {rng.choice([0, 10, 40, 90, 127])} "
                    f"--log2-parts {rng.randint(0, 3)} --key-interval {rng.choice([0, 2, 4])} "
                    f"--segmentation {rng.randint(0, 1)} --lf-deltas {rng.randint(0, 1)} "
                    f"--pct-intra {rng.choice([0, 8, 40, 100])} --pct-split {rng.choice([0, 10, 60])} "
                    f"--pct-new {rng.choice([10, 30])} --pct-skip {rng.choice([0, 35, 90])} "
                    f"--pct-bpred {rng.choice([0, 25, 100])} --coef-density {rng.randint(1, 8)} "
                    f"--pct-empty-block {rng.choice([0, 45, 90])} --golden-period {rng.choice([0, 2, 5])} "
                    f"--altref-period {rng.choice([0, 3, 4])} --hidden-altref {rng.randint(0, 1)}")
    for k in range(40):
        rows = [1, 12, 13, 24, 25][k % 5]
        h = rows * 16 - rng.choice([0, 0, 5, 15])
        w = rng.choice([16, 40, 96, 130, 176])
        parts = 3 if rows == 1 else rng.randint(0, 3)
        cfgs.append(f"--width {w} --height {h} --frames {rng.randint(3, 6)} --seed {2000 + k} "
                    f"--version {rng.randint(0, 3)} --filter-type {rng.randint(0, 1)} --sharpness {rng.choice([0, 3, 7])} "
                    f"--lf {rng.choice([8, 40, 63])} --q {rng.choice([0, 28, 57, 87, 127])} "
                    f"--log2-parts {parts} --key-interval {rng.choice([0, 3])} "
                    f"--segmentation {rng.randint(0, 1)} --lf-deltas {rng.randint(0, 1)} "
                    f"--pct-intra {rng.choice([0, 8, 40, 100])} --pct-split {rng.choice([0, 10, 60])} "
                    f"--pct-new {rng.choice([10, 30, 60])} --pct-skip {rng.choice([0, 35, 90])} "
                    f"--pct-bpred {rng.choice([0, 25, 100])} --coef-density {rng.randint(1, 8)} "
                    f"--pct-empty-block {rng.choice([0, 45, 90])} --golden-period {rng.choice([0, 2, 5])} "
                    f"--altref-period {rng.choice([0, 3, 4])} --hidden-altref {rng.randint(0, 1)} "
                    f"--pct-big-coef {rng.choice([0, 5, 30, 100])} --pct-long-mv {rng.choice([0, 10, 40])} "
                    f"--prob-updates {rng.choice([0, 3, 20])}" + (" --no-skip-flag" if rng.random() < 0.3 else ""))
    return cfgs


# Decode paths of the parity tests: engine settings (read when the engine is created) and how the frames are parsed
# (BatchDecoder's tokens_on_device / device_parse / depth).
DECODE_PATHS = {
    "auto": dict(env={}),
    "swar": dict(env={"VP8R_FILTER": "swar"}),
    "tokens-swar": dict(env={"VP8R_FILTER": "swar"}, tokens_on_device=True),
    "modes-swar": dict(env={"VP8R_FILTER": "swar"}, device_parse=True, depth=3),
    "half-device": dict(env={}, device_parse=0.5),
}


class Engines:
    """One engine per set of engine settings, created on first use (the settings are environment variables the
    engine reads when it is created)."""

    def __init__(self):
        self._by_env = {}

    def get(self, env):
        import vp8_b200
        key = tuple(sorted(env.items()))
        if key not in self._by_env:
            old = os.environ.get("VP8R_FILTER")
            os.environ.pop("VP8R_FILTER", None)
            os.environ.update(env)
            try:
                self._by_env[key] = vp8_b200.Engine(0)
            finally:
                if old is None:
                    os.environ.pop("VP8R_FILTER", None)
                else:
                    os.environ["VP8R_FILTER"] = old
        return self._by_env[key]

    def close(self):
        for e in self._by_env.values():
            e.close()
        self._by_env.clear()


def oracle_frames(payloads):
    """Every frame (shown or not) of one stream through host parser -> oracle: [(I420 bytes, width, height)]."""
    import vp8_b200
    ps, orc = vp8_b200.Parser(), Oracle()
    out = []
    for p in payloads:
        fr = ps.parse(p)
        img = orc.decode(fr)
        d = fr.desc().hdr
        out.append((img, d.width, d.height))
        fr.close()
    orc.close()
    ps.close()
    return out


def oracle_checksums(lib, payloads):
    return [lib.vp8r_checksum_i420(img, w, h) for img, w, h in oracle_frames(payloads)]


def first_difference(got, want, w, h):
    """(plane, x, y) of the first differing byte of two I420 pictures, or None."""
    if got == want:
        return None
    cw, ch = (w + 1) // 2, (h + 1) // 2
    planes = [("Y", 0, w, h), ("U", w * h, cw, ch), ("V", w * h + cw * ch, cw, ch)]
    for i in range(min(len(got), len(want))):
        if got[i] != want[i]:
            for name, at, pw, ph in reversed(planes):
                if i >= at:
                    return name, (i - at) % pw, (i - at) // pw
    return "size", len(got), len(want)


def decode_on_path(engine, payloads, want, path, names, last_frames=None):
    """Decodes the streams `payloads` as one lock-step batch on decode path `path` (a DECODE_PATHS entry) and compares
    every frame's device checksum with `want` (oracle checksums per stream) and, given `last_frames`, each stream's
    last frame byte for byte with last_frames[i].  Returns a list of mismatch descriptions
    naming the stream, the frame and the plane and (x, y) of the first differing sample."""
    import vp8_b200
    bad = []
    dec = vp8_b200.BatchDecoder(engine, len(payloads), pinned=True, tokens_on_device=path.get("tokens_on_device", False),
                                device_parse=path.get("device_parse", False), depth=path.get("depth", 2))

    def on_step(t, live, frames):
        sums = engine.checksum_batch([dec.streams[i] for i in live])
        for i, s in zip(live, sums):
            if s != want[i][t]:
                where = ""
                if len(bad) < 4:  # read the first few back and say where they differ
                    img, w, h = oracle_frames(payloads[i][:t + 1])[t]
                    where = f", first difference (plane, x, y) {first_difference(dec.streams[i].read_frame(), img, w, h)}"
                bad.append(f"{names[i]}: frame {t}{where}")

    dec.decode(payloads, on_step=on_step)
    for i, img in enumerate(last_frames or []):
        if dec.streams[i].read_frame() != img:
            bad.append(f"{names[i]}: last frame differs byte for byte")
    dec.close()
    return bad
