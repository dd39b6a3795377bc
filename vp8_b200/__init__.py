"""vp8_b200: B200-native VP8 frame reconstruction behind the reference decoder's decode surface."""
from .batch import BatchDecoder  # noqa: F401
from . import shard  # noqa: F401
from .decoder import Engine, Parser, ParsedFrame, Stream, decode_ivf, encode_ivf  # noqa: F401
from .ivf import ivf_bytes, read_ivf, write_ivf  # noqa: F401
