"""Loads tests/golden/hap_golden.json (outputs of the unmodified reference, see make_golden.py)."""
import base64
import functools
import hashlib
import json
import os
import zlib

import numpy as np

from hap_b200.abi import (HapTextureFormat_A_RGTC1, HapTextureFormat_RGB_DXT1, HapTextureFormat_RGBA_BPTC_UNORM,
                          HapTextureFormat_RGBA_DXT5, HapTextureFormat_YCoCg_DXT5)

HERE = os.path.dirname(os.path.abspath(__file__))


@functools.lru_cache(None)
def golden():
    with open(os.path.join(HERE, "golden", "hap_golden.json")) as fh:
        return json.load(fh)


def sha(b):
    return hashlib.sha256(bytes(b)).hexdigest()


def b64(s):
    return base64.b64decode(s)


def noise_bytes(n, seed=1):
    import torch
    from hap_b200 import synth
    v = synth.pcg_hash(torch.arange(n, dtype=torch.int64) ^ seed)
    return (v >> 24).to(torch.uint8).numpy().tobytes()


def kat_c_bytes(n=33177600):
    i = np.arange(n, dtype=np.int64)
    return (((i // 4096) * 3) & 0xFF).astype(np.uint8).tobytes()


def pack_frame(frame: bytes) -> str:
    """How hap_golden.json stores a whole frame: zlib, then base64."""
    return base64.b64encode(zlib.compress(bytes(frame), 9)).decode()


def unpack_frame(s: str) -> bytes:
    return zlib.decompress(base64.b64decode(s))


def dxt_like(rng, blocks, bs):
    base = rng.integers(0, 256, size=bs * 8, dtype=np.uint8)
    p = np.tile(base, blocks // 8 + 1)[: blocks * bs].copy()
    p[:: int(rng.integers(5, 60))] = rng.integers(0, 256)
    return p.tobytes()


DIFFERENTIAL_FORMATS = (HapTextureFormat_RGB_DXT1, HapTextureFormat_YCoCg_DXT5, HapTextureFormat_A_RGTC1,
                        HapTextureFormat_RGBA_DXT5, HapTextureFormat_RGBA_BPTC_UNORM)


def block_bytes(fmt):
    return 8 if fmt in (HapTextureFormat_RGB_DXT1, HapTextureFormat_A_RGTC1) else 16


def cpu_differential_case(seed):
    """(payload, format, chunk count) of test_oracle_container.py's seeded differential case `seed`: a half-compressible
    payload of up to 600 blocks."""
    rng = np.random.default_rng(seed)
    blocks = int(rng.integers(1, 600))
    fmt = DIFFERENTIAL_FORMATS[seed % 5]
    bs = block_bytes(fmt)
    base = rng.integers(0, 256, size=bs * 4, dtype=np.uint8)
    payload = np.tile(base, blocks // 4 + 1)[: blocks * bs].copy()
    payload[:: int(rng.integers(3, 50))] = rng.integers(0, 256)
    return payload.tobytes(), fmt, int(rng.integers(1, 12))


def gpu_differential_case(seed):
    """(payload, format, chunk count) of test_gpu_parity.py's seeded differential case `seed`: DXT-like bytes, up to
    40000 blocks."""
    rng = np.random.default_rng(seed)
    fmt = DIFFERENTIAL_FORMATS[seed % 5]
    bs = block_bytes(fmt)
    payload = dxt_like(rng, int(rng.integers(1, 40000)), bs)
    return payload, fmt, int(rng.integers(1, 20))


def container_checks(lib, decode_kw=None):
    """Runs every golden container/Snappy known-answer case against `lib` (a HapABI).  Shared by the
    oracle tests (CPU) and the CUDA library tests (-m gpu).  Returns a list of mismatch strings."""
    from hap_b200.abi import HapCompressorNone, HapCompressorSnappy
    G = golden()
    bad = []
    kw = decode_kw or {}

    def chk(name, got, want):
        if got != want:
            bad.append(f"{name}: got {got!r} want {want!r}")

    # decode of reference frames
    x = bytes([0x55]) * 64
    for key in ("kat_a", "kat_a_none"):
        r, data, fmt, calls = lib.decode(bytes.fromhex(G[key]["frame"]), 0, 64, **kw)
        chk(key + ".decode", (r, data, fmt, calls), (0, x, 0x83F0, []))
    f = bytes.fromhex(G["kat_d"]["frame"])
    chk("kat_d.count", lib.texture_count(f), (0, 2))
    chk("kat_d.formats", [lib.texture_format(f, i)[1] for i in (0, 1)], G["kat_d"]["formats"])
    chk("kat_d.chunks", [lib.chunk_count(f, i)[1] for i in (0, 1)], G["kat_d"]["chunk_counts"])
    r, data, fmt, calls = lib.decode(f, 0, 4096, **kw)
    chk("kat_d.tex0", (r, data, fmt, calls), (0, kat_c_bytes(4096), 0x01, [2]))
    r, data, fmt, calls = lib.decode(f, 1, 2048, **kw)
    chk("kat_d.tex1", (r, data, fmt, calls), (0, bytes([0x55]) * 2048, 0x8DBB, [2]))
    for name, e in G["ref_frames"].items():
        fr = b64(e["frame_b64"])
        if name == "hapm":
            for i in (0, 1):
                r, data, fmt, calls = lib.decode(fr, i, e["payload_len"][i], **kw)
                chk(f"ref_frames.hapm[{i}]", (r, sha(data or b"")), (0, e["payload_sha256"][i]))
        else:
            r, data, fmt, calls = lib.decode(fr, 0, e["payload_len"], **kw)
            chk(f"ref_frames.{name}", (r, sha(data or b""), fmt), (0, e["payload_sha256"], e["format"]))
            chk(f"ref_frames.{name}.chunks", lib.chunk_count(fr, 0), (0, e["chunks"]))
    # raw snappy streams
    for name, e in G["snappy_streams"].items():
        s = bytes.fromhex(e["stream"])
        n = len(s)
        whole = (n.to_bytes(3, "little") + b"\xbe" + s) if n else (b"\0\0\0\xbe" + (0).to_bytes(4, "little"))
        r, data, fmt, calls = lib.decode(whole, 0, 4096, **kw)
        w = e["whole_section"]
        chk(f"snappy.{name}.whole", (r, sha(data) if data is not None else None), (w["result"], w["out_sha256"]))
        di = b"\x01\0\0\x02\x0b" + b"\x04\0\0\x03" + n.to_bytes(4, "little")
        body = len(di).to_bytes(3, "little") + b"\x01" + di + s
        cx = len(body).to_bytes(3, "little") + b"\xce" + body
        r, data, fmt, calls = lib.decode(cx, 0, 4096, **kw)
        w = e["complex_1chunk"]
        chk(f"snappy.{name}.complex", (r, sha(data) if data is not None else None), (w["result"], w["out_sha256"]))
    # container cases
    for name, e in G["container_cases"].items():
        fr = bytes.fromhex(e["frame"])
        r, data, fmt, calls = lib.decode(fr, e["index"], e["cap"], **kw)
        chk(f"case.{name}", (r, data.hex() if data is not None else None, calls), (e["result"], e["out"], e["callback_counts"]))
        if r == 0:
            chk(f"case.{name}.fmt", fmt, e["format"])
        if e["texture_count"] is not None:
            got = lib.texture_count(fr)
            if e["texture_count"][0] == 0:
                chk(f"case.{name}.count", list(got), e["texture_count"])
            else:
                chk(f"case.{name}.count.result", got[0], e["texture_count"][0])
        if e["texture_format"] is not None:
            got = lib.texture_format(fr, e["index"])
            chk(f"case.{name}.format", got[0] if e["texture_format"][0] else list(got), e["texture_format"][0] if e["texture_format"][0] else e["texture_format"])
        if e["chunk_count"] is not None:
            chk(f"case.{name}.chunkcount", list(lib.chunk_count(fr, e["index"])), e["chunk_count"])
    return bad
