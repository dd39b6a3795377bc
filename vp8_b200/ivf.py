"""IVF container demux (32-byte file header, 12-byte frame headers), as src/decode.cc:16-58."""
import struct


def read_ivf(path_or_bytes):
    """Returns (header dict, [frame payload bytes])."""
    data = path_or_bytes if isinstance(path_or_bytes, (bytes, bytearray, memoryview)) else open(path_or_bytes, "rb").read()
    if len(data) < 32 or data[0:4] != b"DKIF":
        raise ValueError("not an IVF file")
    version, hdr_len, fourcc, w, h, rate, scale, n_frames = struct.unpack_from("<HH4sHHIII", data, 4)
    if fourcc != b"VP80":
        raise ValueError(f"unsupported fourcc {fourcc!r}")
    pos = hdr_len
    frames = []
    while pos + 12 <= len(data) and len(frames) < n_frames:
        (size,) = struct.unpack_from("<I", data, pos)
        pos += 12
        frames.append(bytes(data[pos:pos + size]))
        pos += size
    return {"width": w, "height": h, "rate": rate, "scale": scale, "n_frames": n_frames}, frames


def ivf_bytes(width, height, frames, rate=30, scale=1):
    """An IVF file holding `frames` (payload bytes), as bytes."""
    out = [b"DKIF" + struct.pack("<HH4sHHIII", 0, 32, b"VP80", width, height, rate, scale, len(frames)) + b"\0\0\0\0"]
    for i, fr in enumerate(frames):
        out.append(struct.pack("<IQ", len(fr), i))
        out.append(bytes(fr))
    return b"".join(out)


def write_ivf(path, width, height, frames, rate=30, scale=1):
    with open(path, "wb") as f:
        f.write(ivf_bytes(width, height, frames, rate, scale))
