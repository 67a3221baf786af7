"""Pins the CPU oracle (oracle/hap_oracle.c) against the golden vectors produced by the unmodified
reference, and checks the reference build itself against them when it is available."""
import pytest

import oracles
from golden_util import container_checks, cpu_differential_case, golden, kat_c_bytes, noise_bytes, sha, unpack_frame
from hap_b200.abi import (HapCompressorNone, HapCompressorSnappy, HapTextureFormat_A_RGTC1,
                          HapTextureFormat_RGB_DXT1, HapTextureFormat_YCoCg_DXT5)

DXT1, YCOCG, RGTC1 = HapTextureFormat_RGB_DXT1, HapTextureFormat_YCoCg_DXT5, HapTextureFormat_A_RGTC1


def test_oracle_matches_golden_decode_cases():
    assert container_checks(oracles.oracle_abi()) == []


def test_reference_build_matches_its_own_golden():
    ref = oracles.ref_abi()
    if ref is None:
        pytest.skip("reference build unavailable")
    assert container_checks(ref) == []


def test_oracle_encode_kats():
    G = golden()
    o = oracles.oracle_abi()
    x = bytes([0x55]) * 64
    # container bytes are exact; the Snappy payload of these tiny inputs also matches Google's bytes
    assert o.encode([x], [DXT1], [HapCompressorSnappy], [1])[1].hex() == G["kat_a"]["frame"]
    assert o.encode([x], [DXT1], [HapCompressorNone], [1])[1].hex() == G["kat_a_none"]["frame"]
    assert o.max_encoded_length([64], [DXT1], [1]) == G["kat_a"]["max_len"]
    assert o.max_encoded_length([1036800], [DXT1], [1]) == G["max_len_1080p_dxt1"] == 1209665
    r, f = o.encode([kat_c_bytes(4096), bytes([0x55]) * 2048], [YCOCG, RGTC1], [1, 1], [2, 2])
    assert f.hex() == G["kat_d"]["frame"]
    assert o.max_encoded_length([4096, 2048], [YCOCG, RGTC1], [2, 2]) == G["kat_d"]["max_len"]
    r, f = o.encode([kat_c_bytes(4096), bytes([0x55]) * 2048], [YCOCG, RGTC1], [0, 0], [2, 2])
    assert (sha(f), len(f), f[:12].hex()) == (G["kat_d_none"]["frame_sha256"], G["kat_d_none"]["frame_len"], G["kat_d_none"]["header"])


def test_oracle_whole_frame_fallback_kat_b():
    G = golden()["kat_b"]
    nb = noise_bytes(4147200)
    assert sha(nb) == G["input_sha256"]
    r, f = oracles.oracle_abi().encode([nb], [DXT1], [HapCompressorSnappy], [4])
    assert r == 0 and len(f) == G["frame_len"] and sha(f) == G["frame_sha256"]


def test_oracle_eight_byte_header_kat_c():
    G = golden()["kat_c"]
    o = oracles.oracle_abi()
    cb = kat_c_bytes()
    assert sha(cb) == G["input_sha256"]
    r, f = o.encode([cb], [YCOCG], [HapCompressorSnappy], [8])
    assert r == 0
    # header, DI container and compressor table are exact; chunk sizes depend on the Snappy encoder
    assert f[:28].hex() == G["header"][:56].replace(G["header"][8:16], f[4:8].hex())
    assert f[:4].hex() == "000000cf"
    assert o.max_encoded_length([len(cb)], [YCOCG], [8]) == G["max_len"]
    assert o.decode(f, 0, len(cb) - 1)[0] == G["results"]["short_out"]
    assert o.decode(f[:-5], 0, len(cb))[0] == G["results"]["truncated_in"]
    assert o.decode(f, 1, len(cb))[0] == G["results"]["index_1"]
    assert o.decode(f, 0, len(cb), callback=None)[0] == G["results"]["null_callback"]
    r, data, fmt, calls = o.decode(f, 0, len(cb))
    assert r == 0 and data == cb and calls == G["callback_counts"]


def test_oracle_chunk_limiter_kat_e():
    G = golden()["kat_e"]
    o = oracles.oracle_abi()
    payload = kat_c_bytes(1036800)
    for ask, e in G.items():
        r, f = o.encode([payload], [DXT1], [HapCompressorSnappy], [int(ask)])
        assert r == e["result"]
        assert o.chunk_count(f, 0)[1] == e["chunk_count"], ask
        assert f[3] == e["type"], ask
    assert oracles.limited_chunk_count(1036800, DXT1, 7) == 6
    assert oracles.limited_chunk_count(1036800, DXT1, 11) == 10
    assert oracles.limited_chunk_count(1036800, DXT1, 1000) == 960


def test_oracle_encode_argument_results():
    G = golden()["encode_results"]
    o = oracles.oracle_abi()
    p16 = bytes(16)
    assert o.encode([p16], [DXT1], [1], [0])[0] == G["chunk_0"]
    assert o.encode([p16], [0x1234], [1], [1])[0] == G["bad_format"]
    assert o.encode([p16], [DXT1], [7], [1])[0] == G["bad_compressor"]
    assert o.encode([p16], [DXT1], [1], [1], out_capacity=20)[0] == G["small_buffer"]
    assert o.encode([p16, p16], [DXT1, DXT1], [1, 1], [1, 1])[0] == G["two_dxt1"]
    assert o.encode([p16, p16], [YCOCG, DXT1], [1, 1], [1, 1])[0] == G["ycocg_plus_dxt1"]


@pytest.mark.parametrize("seed", range(6))
def test_oracle_vs_reference_differential(seed):
    """Random payloads/chunk counts against the reference's frames of them (golden): None frames byte-identical; Snappy
    frames cross-decode."""
    G = golden()["differential_cpu"][str(seed)]
    o = oracles.oracle_abi()
    payload, fmt, k = cpu_differential_case(seed)
    assert o.max_encoded_length([len(payload)], [fmt], [k]) == G["max_len"]
    on, fo = o.encode([payload], [fmt], [HapCompressorNone], [k])
    assert (on, len(fo), sha(fo)) == (G["none"]["result"], G["none"]["frame_len"], G["none"]["frame_sha256"])
    fs = unpack_frame(G["snappy"]["frame"])
    os_, fo = o.encode([payload], [fmt], [HapCompressorSnappy], [k])
    assert G["snappy"]["result"] == os_ == 0
    assert list(o.chunk_count(fo, 0)) == G["snappy"]["chunk_count"]
    # the reference decoded this very oracle frame to the payload
    assert sha(fo) == G["oracle_snappy_frame"]["frame_sha256"]
    assert G["oracle_snappy_frame"]["reference_decode"] == [0, sha(payload), fmt]
    assert o.decode(fs, 0, len(payload))[:3] == (0, payload, fmt)
