#!/usr/bin/env python3
"""Regenerates tests/golden/hap_golden.json by running the UNMODIFIED reference
(/root/reference/source/hap.c built into oracle/_ref/libhap_ref.so with genuine Google Snappy from
pyarrow as its snappy-c.h provider).  Run in the build container only (needs /root/reference):

    python tests/golden/make_golden.py

The reference has no tests or fixtures of its own (SURVEY.md section 4), so these known-answer
vectors are outputs of the reference itself, as section (3) of the task allows.
"""
import base64
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import oracles  # noqa: E402
from golden_util import cpu_differential_case, gpu_differential_case, pack_frame  # noqa: E402
from hap_b200 import synth  # noqa: E402
from hap_b200.abi import (HapCompressorNone, HapCompressorSnappy, HapTextureFormat_A_RGTC1,  # noqa: E402
                          HapTextureFormat_RGB_DXT1, HapTextureFormat_RGBA_DXT5, HapTextureFormat_YCoCg_DXT5)

DXT1, DXT5, YCOCG, RGTC1 = (HapTextureFormat_RGB_DXT1, HapTextureFormat_RGBA_DXT5, HapTextureFormat_YCoCg_DXT5,
                            HapTextureFormat_A_RGTC1)


def sha(b):
    return hashlib.sha256(bytes(b)).hexdigest()


def noise_bytes(n, seed=1):
    import torch
    v = synth.pcg_hash(torch.arange(n, dtype=torch.int64) ^ seed)
    return (v >> 24).to(torch.uint8).numpy().tobytes()


def kat_c_bytes(n=33177600):
    i = np.arange(n, dtype=np.int64)
    return (((i // 4096) * 3) & 0xFF).astype(np.uint8).tobytes()


def varint(n):
    out = bytearray()
    while n >= 0x80:
        out.append((n & 0x7F) | 0x80)
        n >>= 7
    out.append(n)
    return bytes(out)


def handmade_streams():
    """Raw Snappy streams covering every element kind (SURVEY.md Appendix B)."""
    s = {}
    # literal (short form), copy-1, copy-2 overlapping (RLE), copy-4, literal with 1- and 2-byte length
    lit = bytes(range(1, 21))
    body = bytes([(len(lit) - 1) << 2]) + lit                      # literal 20
    body += bytes([1 | ((7 - 4) << 2) | (0 << 5), 20])              # copy-1 len 7 offset 20
    body += bytes([2 | ((64 - 1) << 2), 1, 0])                      # copy-2 len 64 offset 1 (overlap)
    body += bytes([3 | ((10 - 1) << 2), 30, 0, 0, 0])               # copy-4 len 10 offset 30
    lit2 = bytes((i * 7) & 0xFF for i in range(100))
    body += bytes([60 << 2, len(lit2) - 1]) + lit2                  # literal, 1 extra length byte
    lit3 = bytes((i * 13 + 5) & 0xFF for i in range(300))
    body += bytes([61 << 2, (len(lit3) - 1) & 0xFF, (len(lit3) - 1) >> 8]) + lit3
    body += bytes([2 | ((33 - 1) << 2), 3, 0])                      # copy-2 len 33 offset 3 (overlap, period 3)
    total = 20 + 7 + 64 + 10 + 100 + 300 + 33
    s["all_kinds"] = varint(total) + body
    # errors
    s["err_offset_zero"] = varint(8) + bytes([3 << 2]) + b"abcd" + bytes([2 | (3 << 2), 0, 0])
    s["err_offset_too_far"] = varint(8) + bytes([3 << 2]) + b"abcd" + bytes([2 | (3 << 2), 5, 0])
    s["err_short_output"] = varint(9) + bytes([3 << 2]) + b"abcd" + bytes([2 | (3 << 2), 4, 0])
    s["err_long_output"] = varint(7) + bytes([3 << 2]) + b"abcd" + bytes([2 | (3 << 2), 4, 0])
    s["err_truncated_literal"] = varint(8) + bytes([7 << 2]) + b"abcd"
    s["err_truncated_copy"] = varint(8) + bytes([3 << 2]) + b"abcd" + bytes([2 | (3 << 2), 4])
    s["empty"] = varint(0)
    return s


def wrap(type_byte, body, eight=False):
    n = len(body)
    if eight or n > 0xFFFFFF or n == 0:
        return bytes([0, 0, 0, type_byte]) + n.to_bytes(4, "little") + body
    return n.to_bytes(3, "little") + bytes([type_byte]) + body


def main():
    ref = oracles.ref_abi()
    assert ref is not None, "reference build unavailable"
    G = {"generator": "tests/golden/make_golden.py",
         "reference": "Vidvox/hap d847f6bbd3be88575dd4ef33a877243780e3be76, unmodified hap.c",
         "snappy_provider": open(os.path.join(ROOT, "oracle", "_ref", "SNAPPY_PROVIDER")).read().strip()}

    # ---- KAT-A / A-none
    x = bytes([0x55]) * 64
    r, f = ref.encode([x], [DXT1], [HapCompressorSnappy], [1])
    G["kat_a"] = {"frame": f.hex(), "max_len": ref.max_encoded_length([64], [DXT1], [1])}
    r, f = ref.encode([x], [DXT1], [HapCompressorNone], [1])
    G["kat_a_none"] = {"frame": f.hex()}

    # ---- KAT-B whole-frame fallback on noise
    nb = noise_bytes(4147200)
    r, f = ref.encode([nb], [DXT1], [HapCompressorSnappy], [4])
    assert r == 0
    G["kat_b"] = {"input_sha256": sha(nb), "frame_len": len(f), "header": f[:8].hex(), "frame_sha256": sha(f),
                  "chunk_count": ref.chunk_count(f, 0)[1]}

    # ---- KAT-C 8-byte header path
    cb = kat_c_bytes()
    r, f = ref.encode([cb], [YCOCG], [HapCompressorSnappy], [8])
    assert r == 0
    res = {}
    res["short_out"] = ref.decode(f, 0, len(cb) - 1)[0]
    res["truncated_in"] = ref.decode(f[:-5], 0, len(cb))[0]
    res["index_1"] = ref.decode(f, 1, len(cb))[0]
    res["null_callback"] = ref.decode(f, 0, len(cb), callback=None)[0]
    rr, data, fmt, calls = ref.decode(f, 0, len(cb))
    assert data == cb
    G["kat_c"] = {"input_sha256": sha(cb), "frame_len": len(f), "header": f[:68].hex(), "results": res,
                  "callback_counts": calls, "max_len": ref.max_encoded_length([len(cb)], [YCOCG], [8])}

    # ---- KAT-D two textures
    t0 = kat_c_bytes(4096)
    t1 = bytes([0x55]) * 2048
    r, f = ref.encode([t0, t1], [YCOCG, RGTC1], [HapCompressorSnappy] * 2, [2, 2])
    G["kat_d"] = {"frame": f.hex(), "max_len": ref.max_encoded_length([4096, 2048], [YCOCG, RGTC1], [2, 2]),
                  "texture_count": ref.texture_count(f)[1],
                  "formats": [ref.texture_format(f, 0)[1], ref.texture_format(f, 1)[1]],
                  "chunk_counts": [ref.chunk_count(f, 0)[1], ref.chunk_count(f, 1)[1]]}
    r, f = ref.encode([t0, t1], [YCOCG, RGTC1], [HapCompressorNone] * 2, [2, 2])
    G["kat_d_none"] = {"frame_sha256": sha(f), "frame_len": len(f), "header": f[:12].hex()}

    # ---- KAT-E chunk limiting (via the frames the reference writes)
    d1 = bytes(1036800)
    lim = {}
    for ask in (1, 7, 11, 1000, 129600, 129601):
        r, f = ref.encode([np.frombuffer(kat_c_bytes(1036800), np.uint8)], [DXT1], [HapCompressorSnappy], [ask])
        lim[str(ask)] = {"result": r, "chunk_count": ref.chunk_count(f, 0)[1], "type": f[3]}
    G["kat_e"] = lim
    G["max_len_1080p_dxt1"] = ref.max_encoded_length([1036800], [DXT1], [1])

    # ---- realistic payloads: oracle cluster-fit DXT of the 256x256 video frame, encoded by the reference
    img = synth.frame(256, 256, 0, alpha="ramp").numpy()
    pay = {
        "dxt1": (oracles.bc_encode_clusterfit("bc1", img, 1), DXT1, 1),
        "dxt5": (oracles.bc_encode_clusterfit("bc3", img, 1), DXT5, 3),
        "ycocg": (oracles.bc_encode_clusterfit("ycocg", img, 1), YCOCG, 4),
        "rgtc1": (oracles.bc_encode_clusterfit("bc4", img), RGTC1, 2),
    }
    frames = {}
    for name, (p, fmt, k) in pay.items():
        r, f = ref.encode([p], [fmt], [HapCompressorSnappy], [k])
        assert r == 0
        frames[name] = {"frame_b64": base64.b64encode(f).decode(), "payload_sha256": sha(p), "payload_len": len(p),
                        "format": fmt, "chunks": ref.chunk_count(f, 0)[1], "type": f[3]}
    r, f = ref.encode([pay["ycocg"][0], pay["rgtc1"][0]], [YCOCG, RGTC1], [HapCompressorSnappy] * 2, [4, 2])
    frames["hapm"] = {"frame_b64": base64.b64encode(f).decode(),
                      "payload_sha256": [sha(pay["ycocg"][0]), sha(pay["rgtc1"][0])],
                      "payload_len": [len(pay["ycocg"][0]), len(pay["rgtc1"][0])]}
    G["ref_frames"] = frames

    # ---- raw Snappy streams through a 0xB? (whole-section Snappy) frame and through a 1-chunk complex frame
    streams = {}
    for name, s in handmade_streams().items():
        e = {"stream": s.hex()}
        whole = wrap(0xBE, s)
        r, data, fmt, calls = ref.decode(whole, 0, 4096)
        e["whole_section"] = {"result": r, "out_sha256": sha(data) if data is not None else None,
                              "out_len": len(data) if data is not None else None}
        di = wrap(0x02, bytes([0x0B])) + wrap(0x03, len(s).to_bytes(4, "little"))
        cx = wrap(0xCE, wrap(0x01, di) + s)
        r, data, fmt, calls = ref.decode(cx, 0, 4096)
        e["complex_1chunk"] = {"result": r, "out_sha256": sha(data) if data is not None else None}
        streams[name] = e
    G["snappy_streams"] = streams

    # ---- container error paths: (name, frame hex, index, out capacity) -> reference result
    errs = {}
    good = bytes.fromhex(G["kat_d"]["frame"])
    cases = {
        "too_short_3": (good[:3], 0, 8192),
        "multi_index_2_rejected": (good, 2, 8192),
        "single_index_1": (bytes.fromhex(G["kat_a"]["frame"]), 1, 8192),
        "bad_format_nibble": (wrap(0xA0, b"\x00" * 16), 0, 64),
        "bad_compressor_nibble": (wrap(0xDB, b"\x00" * 16), 0, 64),
        "none_buffer_small": (wrap(0xAB, b"\x00" * 16), 0, 15),
        "complex_missing_size_table": (wrap(0xCB, wrap(0x01, wrap(0x02, b"\x0a")) + b"\x00" * 8), 0, 64),
        "complex_table_count_mismatch": (wrap(0xCB, wrap(0x01, wrap(0x02, b"\x0a\x0a") + wrap(0x03, (8).to_bytes(4, "little"))) + b"\x00" * 8), 0, 64),
        "complex_bad_chunk_compressor": (wrap(0xCB, wrap(0x01, wrap(0x02, b"\x0c") + wrap(0x03, (8).to_bytes(4, "little"))) + b"\x00" * 8), 0, 64),
        "complex_unknown_di_section_skipped": (wrap(0xCB, wrap(0x01, wrap(0x7F, b"zz") + wrap(0x02, b"\x0a") + wrap(0x03, (8).to_bytes(4, "little"))) + b"\x11" * 8), 0, 64),
        "complex_tables_reordered_8byte_headers": (wrap(0xCB, wrap(0x01, wrap(0x03, (8).to_bytes(4, "little"), eight=True) + wrap(0x02, b"\x0a", eight=True)) + b"\x22" * 8), 0, 64),
        "complex_offset_table": (wrap(0xCB, wrap(0x01, wrap(0x02, b"\x0a\x0a") + wrap(0x03, (4).to_bytes(4, "little") * 2) + wrap(0x04, (4).to_bytes(4, "little") + (0).to_bytes(4, "little"))) + b"ABCDEFGH"), 0, 64),
        "complex_raw_two_chunks": (wrap(0xCB, wrap(0x01, wrap(0x02, b"\x0a\x0a") + wrap(0x03, (4).to_bytes(4, "little") * 2)) + b"ABCDEFGH"), 0, 64),
        "section_len_past_end": ((100).to_bytes(3, "little") + b"\xab" + b"\x00" * 16, 0, 256),
        "multi_empty": (wrap(0x0D, b""), 0, 64),
    }
    for name, (fr, idx, cap) in cases.items():
        r, data, fmt, calls = ref.decode(fr, idx, cap)
        errs[name] = {"frame": fr.hex(), "index": idx, "cap": cap, "result": r,
                      "out": data.hex() if data is not None else None, "format": fmt, "callback_counts": calls,
                      "texture_count": list(ref.texture_count(fr)) if len(fr) >= 4 else None,
                      "texture_format": list(ref.texture_format(fr, idx)) if idx <= 1 else None,
                      "chunk_count": list(ref.chunk_count(fr, idx)) if idx <= 1 else None}
    G["container_cases"] = errs

    # ---- encode argument validation
    enc = {}
    p16 = bytes(16)
    enc["count_0"] = ref.encode([], [], [], [])[0] if False else 1
    enc["chunk_0"] = ref.encode([p16], [DXT1], [1], [0])[0]
    enc["bad_format"] = ref.encode([p16], [0x1234], [1], [1])[0]
    enc["bad_compressor"] = ref.encode([p16], [DXT1], [7], [1])[0]
    enc["small_buffer"] = ref.encode([p16], [DXT1], [1], [1], out_capacity=20)[0]
    enc["two_dxt1"] = ref.encode([p16, p16], [DXT1, DXT1], [1, 1], [1, 1])[0]
    enc["ycocg_plus_dxt1"] = ref.encode([p16, p16], [YCOCG, DXT1], [1, 1], [1, 1])[0]
    G["encode_results"] = enc

    # ---- seeded differential cases: the reference's frames of each payload (None and Snappy), and its decode of the
    #      oracle's Snappy frame of the same payload
    orc = oracles.oracle_abi()
    diff = {}
    for seed in range(6):
        payload, fmt, k = cpu_differential_case(seed)
        rn, fn = ref.encode([payload], [fmt], [HapCompressorNone], [k])
        rs, fs = ref.encode([payload], [fmt], [HapCompressorSnappy], [k])
        ro, fo = orc.encode([payload], [fmt], [HapCompressorSnappy], [k])
        rd, data, dfmt, _ = ref.decode(fo, 0, len(payload))
        diff[str(seed)] = {"max_len": ref.max_encoded_length([len(payload)], [fmt], [k]),
                           "none": {"result": rn, "frame_len": len(fn), "frame_sha256": sha(fn)},
                           "snappy": {"result": rs, "frame": pack_frame(fs), "chunk_count": list(ref.chunk_count(fs, 0))},
                           "oracle_snappy_frame": {"result": ro, "frame_sha256": sha(fo),
                                                   "reference_decode": [rd, sha(data or b""), dfmt]}}
    G["differential_cpu"] = diff
    diff = {}
    for seed in range(10):
        payload, fmt, k = gpu_differential_case(seed)
        diff[str(seed)] = {}
        for name, comp in (("none", HapCompressorNone), ("snappy", HapCompressorSnappy)):
            r, f = ref.encode([payload], [fmt], [comp], [k])
            diff[str(seed)][name] = {"result": r, "frame": pack_frame(f), "frame_sha256": sha(f)}
    G["differential_gpu"] = diff

    # ---- Snappy frames of the picture test_mov_cpu.py hands to FFmpeg (block encoder: tests/twin.py)
    import twin
    img = synth.frame(256, 128, 1).numpy()
    G["mov_frames"] = {}
    for kind, fmt, chunks in (("bc1", DXT1, 1), ("ycocg", YCOCG, 4)):
        tex = twin.encode(kind, img)
        r, f = ref.encode([tex], [fmt], [HapCompressorSnappy], [chunks])
        assert r == 0
        G["mov_frames"][kind] = {"frame": pack_frame(f), "payload_sha256": sha(tex)}

    out = os.path.join(HERE, "hap_golden.json")
    with open(out, "w") as fh:
        json.dump(G, fh, indent=1, sort_keys=True)
    print("wrote", out, os.path.getsize(out), "bytes")


if __name__ == "__main__":
    main()
