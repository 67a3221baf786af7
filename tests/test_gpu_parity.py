"""Parity of the CUDA path (libhap_b200.so, through its C-ABI) against the reference: golden vectors
produced by the unmodified hap.c, the CPU oracle on seeded inputs, and size-independent round-trip
properties at BASELINE.json's full sizes.  Bit-exact throughout (byte work)."""
import numpy as np
import pytest
import torch

import hap_b200
import oracles
from golden_util import container_checks, dxt_like, golden, gpu_differential_case, kat_c_bytes, noise_bytes, sha, unpack_frame
from hap_b200 import synth
from hap_b200.abi import (HapCompressorNone, HapCompressorSnappy, HapTextureFormat_A_RGTC1, HapTextureFormat_RGB_DXT1,
                          HapTextureFormat_YCoCg_DXT5)

pytestmark = pytest.mark.gpu
DXT1, YCOCG, RGTC1 = HapTextureFormat_RGB_DXT1, HapTextureFormat_YCoCg_DXT5, HapTextureFormat_A_RGTC1


@pytest.fixture(scope="module")
def lib():
    return hap_b200.load()


def test_golden_vectors_of_the_reference(lib):
    assert container_checks(lib) == []


def test_kernels_really_ran(lib):
    before = lib.launches()
    x = bytes([0x55]) * 64
    r, f = lib.encode([x], [DXT1], [HapCompressorSnappy], [1])
    assert r == 0 and lib.launches() >= before + 3
    assert lib.decode(f, 0, 64)[:3] == (0, x, DXT1)
    assert lib.launches() >= before + 4


def test_encode_kats(lib):
    G = golden()
    orc = oracles.oracle_abi()
    x = bytes([0x55]) * 64
    r, f = lib.encode([x], [DXT1], [HapCompressorSnappy], [1])
    # container bytes up to the size table are fixed by the format; the Snappy bytes are ours
    assert r == 0 and f[3] == 0xCB and f[4:17].hex() == G["kat_a"]["frame"][8:34]
    assert orc.decode(f, 0, 64)[:3] == (0, x, DXT1)
    # KAT-B: incompressible -> whole-texture fallback, byte-identical to the reference
    nb = noise_bytes(4147200)
    r, f = lib.encode([nb], [DXT1], [HapCompressorSnappy], [4])
    assert r == 0 and len(f) == G["kat_b"]["frame_len"] and sha(f) == G["kat_b"]["frame_sha256"]
    # KAT-C: 8-byte header chosen before compression
    cb = kat_c_bytes()
    r, f = lib.encode([cb], [YCOCG], [HapCompressorSnappy], [8])
    assert r == 0 and f[:4].hex() == "000000cf" and f[8:28].hex() == G["kat_c"]["header"][16:56]
    assert lib.chunk_count(f, 0) == (0, 8)
    assert lib.decode(f, 0, len(cb) - 1)[0] == G["kat_c"]["results"]["short_out"]
    assert lib.decode(f[:-5], 0, len(cb))[0] == G["kat_c"]["results"]["truncated_in"]
    r, data, fmt, calls = lib.decode(f, 0, len(cb))
    assert r == 0 and data == cb and calls == [8]
    assert orc.decode(f, 0, len(cb))[:2] == (0, cb)
    # KAT-D: two textures
    t0, t1 = kat_c_bytes(4096), bytes([0x55]) * 2048
    r, f = lib.encode([t0, t1], [YCOCG, RGTC1], [1, 1], [2, 2])
    assert r == 0 and lib.texture_count(f) == (0, 2)
    assert orc.decode(f, 0, 4096)[:3] == (0, t0, YCOCG) and orc.decode(f, 1, 2048)[:3] == (0, t1, RGTC1)
    # KAT-E: chunk limiting
    payload = kat_c_bytes(1036800)
    for ask, e in G["kat_e"].items():
        r, f = lib.encode([payload], [DXT1], [HapCompressorSnappy], [int(ask)])
        assert r == e["result"] and lib.chunk_count(f, 0)[1] == e["chunk_count"] and f[3] == e["type"], ask


@pytest.mark.parametrize("seed", range(10))
def test_differential_against_oracle_and_reference(lib, seed):
    payload, fmt, k = gpu_differential_case(seed)
    G = golden()["differential_gpu"][str(seed)]
    orc, ref = oracles.oracle_abi(), oracles.ref_abi()
    for comp, name in ((HapCompressorNone, "none"), (HapCompressorSnappy, "snappy")):
        r, f = lib.encode([payload], [fmt], [comp], [k])
        assert r == 0
        ro, fo = orc.encode([payload], [fmt], [comp], [k])
        if comp == HapCompressorNone:
            assert f == fo and sha(f) == G[name]["frame_sha256"]      # byte-identical to the reference's frame
        assert lib.chunk_count(f, 0) == orc.chunk_count(fo, 0)
        for dec in (orc, ref, lib):       # ref: the reference build, where it has been built
            if dec is not None:
                assert dec.decode(f, 0, len(payload))[:3] == (0, payload, fmt)
        # frames compressed by the oracle and (golden) by Google Snappy through the reference decode on the GPU
        assert lib.decode(fo, 0, len(payload))[:3] == (0, payload, fmt)
        fr = unpack_frame(G[name]["frame"])
        assert G[name]["result"] == 0 and sha(fr) == G[name]["frame_sha256"]
        assert lib.decode(fr, 0, len(payload))[:3] == (0, payload, fmt)


def test_corrupt_streams_never_crash_and_match_oracle_status(lib):
    rng = np.random.default_rng(5)
    orc = oracles.oracle_abi()
    payload = dxt_like(rng, 5000, 16)
    r, good = orc.encode([payload], [YCOCG], [1], [3])
    for i in range(60):
        f = bytearray(good)
        what = i % 3
        if what == 0:
            f = f[: len(f) - 1 - int(rng.integers(0, 300))]
        elif what == 1:
            f[int(rng.integers(4, len(f)))] ^= 1 << int(rng.integers(0, 8))
        else:
            p = int(rng.integers(40, len(f) - 2))
            f[p] = int(rng.integers(0, 256))
        f = bytes(f)
        want = orc.decode(f, 0, len(payload))
        got = lib.decode(f, 0, len(payload))
        if want[0] == 0:
            assert got[:3] == want[:3], i
        else:
            # the oracle may run off the section like hap.c does (SURVEY.md Q9); ours must say Bad_Frame or agree
            assert got[0] != 0, i


def test_device_pointers_and_callback_contract(lib):
    rng = np.random.default_rng(9)
    payload = dxt_like(rng, 8192, 16)
    r, f = lib.encode([payload], [YCOCG], [1], [8])
    dev_frame = torch.frombuffer(bytearray(f), dtype=torch.uint8).cuda()
    dev_out = torch.empty(len(payload), dtype=torch.uint8, device="cuda")
    r, used, fmt, calls = lib.decode((dev_frame.data_ptr(), len(f)), 0, len(payload), out=(dev_out.data_ptr(), len(payload)))
    assert (r, used, fmt, calls) == (0, len(payload), YCOCG, [8])
    assert dev_out.cpu().numpy().tobytes() == payload
    # one chunk: the callback must not be called
    r, f1 = lib.encode([payload], [YCOCG], [1], [1])
    assert lib.decode(f1, 0, len(payload))[3] == []
    # device texture in, device frame out
    dev_tex = torch.frombuffer(bytearray(payload), dtype=torch.uint8).cuda()
    cap = lib.max_encoded_length([len(payload)], [YCOCG], [8])
    dev_f = torch.empty(cap, dtype=torch.uint8, device="cuda")
    r, used = lib.encode([(dev_tex.data_ptr(), len(payload))], [YCOCG], [1], [8], out=(dev_f.data_ptr(), cap), out_capacity=cap)
    assert r == 0 and dev_f[:used].cpu().numpy().tobytes() == f


def test_device_frame_header_walks_fetch_pages_only(lib):
    """Queries and HapDecode on a DEVICE frame read headers through a lazily fetched mirror (hap_api.cu HeaderView): a
    two-texture frame whose second section header, tables and chunk heads lie megabytes apart must give exactly what the
    same calls give on the host copy of the frame, for both textures, with and without the trailing index."""
    rng = np.random.default_rng(21)
    t0 = dxt_like(rng, 65536, 16)          # 1 MiB colour plane
    t1 = dxt_like(rng, 65536, 8)           # 512 KiB alpha plane
    for write_index in (1, 0):
        lib.set_option(lib.OPTION_WRITE_INDEX, write_index)
        try:
            r, f = lib.encode([t0, t1], [YCOCG, RGTC1], [1, 1], [16, 8])
        finally:
            lib.set_option(lib.OPTION_WRITE_INDEX, 1)
        assert r == 0
        dev = torch.frombuffer(bytearray(f), dtype=torch.uint8).cuda()
        dp = (dev.data_ptr(), len(f))
        assert lib.texture_count(dp) == lib.texture_count(f) == (0, 2)
        for i, (t, fmt, k) in enumerate(((t0, YCOCG, 16), (t1, RGTC1, 8))):
            assert lib.texture_format(dp, i) == lib.texture_format(f, i) == (0, fmt)
            assert lib.chunk_count(dp, i) == lib.chunk_count(f, i) == (0, k)
            out = torch.zeros(len(t), dtype=torch.uint8, device="cuda")
            r, used, gf, calls = lib.decode(dp, i, len(t), out=(out.data_ptr(), len(t)))
            assert (r, used, gf, calls) == (0, len(t), fmt, [k])
            assert out.cpu().numpy().tobytes() == t
            assert lib.decode(dp, i, len(t))[:3] == (0, t, fmt)          # device frame, host texture
        # a truncated device frame fails like its host copy does
        for cut in (3, 9, 4099, len(f) // 2):
            assert lib.decode((dev.data_ptr(), cut), 1, len(t1))[0] == lib.decode(f[:cut], 1, len(t1))[0] != 0


def test_delivery_ring_on_one_device(lib):
    """HapB200Ring* with producer and consumer on the same GPU: frames encoded straight into the ring are the frames a
    plain batch encode writes; flags order the consumer behind the producer; bad arguments are refused."""
    from hap_b200.lib import HapB200Codec_HapM
    w, h, k, n = 256, 128, 4, 3
    dev = torch.device("cuda", torch.cuda.current_device())
    imgs = torch.stack([synth.frame(w, h, i, alpha="ramp", device="cuda") for i in range(n)])
    cap = (lib.max_encoded_length_rgba(w, h, HapB200Codec_HapM, k) + 255) // 256 * 256
    plain = torch.zeros((n, cap), dtype=torch.uint8, device="cuda")
    used = torch.zeros(n, dtype=torch.int64, device="cuda")
    assert lib.encode_rgba_batch(imgs.data_ptr(), n, w * h * 4, w, h, HapB200Codec_HapM, 1, k, plain.data_ptr(), cap, used.data_ptr()) == 0
    header = 4096
    r, ring, handle = lib.ring_create(dev.index, header + n * cap)
    assert r == 0 and ring != 0 and len(handle) == lib.RING_HANDLE_BYTES
    try:
        producer, consumer = torch.cuda.Stream(), torch.cuda.Stream()
        got = torch.zeros((n, cap), dtype=torch.uint8, device="cuda")
        glen = torch.zeros(n, dtype=torch.int64, device="cuda")
        torch.cuda.synchronize()
        # queued BEFORE the producer runs: the polling kind of wait (it ends by itself; on ONE device a wait that is ahead of
        # the work it waits for can hold that work back when the two streams share a hardware queue -- include/hap_b200.h)
        assert lib.ring_wait(dev.index, ring, 1, 3000, stream=consumer.cuda_stream) == 0

        class _Ext:
            def __init__(self, ptr, nb):
                self.__cuda_array_interface__ = {"shape": (nb,), "typestr": "|u1", "data": (ptr, False), "version": 2}
        ring_t = torch.as_tensor(_Ext(ring, header + n * cap), device="cuda")
        with torch.cuda.stream(consumer):
            got.copy_(ring_t[header:].view(n, cap))
            glen.copy_(ring_t[64: 64 + 8 * n].view(torch.int64))
        assert lib.encode_rgba_batch(imgs.data_ptr(), n, w * h * 4, w, h, HapB200Codec_HapM, 1, k, ring + header, cap, ring + 64,
                                     stream=producer.cuda_stream) == 0
        assert lib.ring_publish(dev.index, ring, 1, stream=producer.cuda_stream) == 0
        consumer.synchronize()
        assert lib.ring_wait(dev.index, ring, 1, 0, stream=consumer.cuda_stream) == 0       # published already: the stream memory operation passes
        consumer.synchronize()
        if not torch.equal(glen, used):         # (the first wait timed out before the producer got to run: read again)
            with torch.cuda.stream(consumer):
                got.copy_(ring_t[header:].view(n, cap))
                glen.copy_(ring_t[64: 64 + 8 * n].view(torch.int64))
            consumer.synchronize()
        assert torch.equal(glen, used)
        for i in range(n):
            assert torch.equal(got[i, : int(used[i])], plain[i, : int(used[i])])
        del ring_t
        # refused: misaligned flag, no flag, device out of range
        assert lib.ring_publish(dev.index, ring + 2, 1) != 0 and lib.ring_wait(dev.index, 0, 1, 10) != 0
        assert lib.ring_create(99, 4096)[0] != 0 and lib.ring_attach(dev.index, 99) != 0 and lib.ring_attach(dev.index, dev.index) == 0
    finally:
        assert lib.ring_destroy(dev.index, ring) == 0


def test_batch_encode_decode_roundtrip(lib):
    from hap_b200.lib import HapB200Codec_HapY
    frames, n = 6, 16 * 4096
    rng = np.random.default_rng(11)
    tex = torch.frombuffer(bytearray(b"".join(dxt_like(rng, 4096, 16) for _ in range(frames))), dtype=torch.uint8).cuda()
    cap = (lib.max_encoded_length([n], [YCOCG], [4]) + 15) // 16 * 16
    out = torch.zeros(frames * cap, dtype=torch.uint8, device="cuda")
    used = torch.zeros(frames, dtype=torch.int64, device="cuda")
    assert lib.encode_batch([tex.data_ptr()], [n], [n], [YCOCG], [1], [4], frames, out.data_ptr(), cap, used.data_ptr()) == 0
    orc = oracles.oracle_abi()
    host = out.cpu().numpy()
    for f in range(frames):
        fr = host[f * cap: f * cap + int(used[f])].tobytes()
        assert orc.decode(fr, 0, n)[:2] == (0, tex[f * n:(f + 1) * n].cpu().numpy().tobytes())
    back = torch.zeros(frames * n, dtype=torch.uint8, device="cuda")
    bused = torch.zeros(frames, dtype=torch.int64, device="cuda")
    fmts = torch.zeros(frames, dtype=torch.int32, device="cuda")
    res = torch.full((frames,), 77, dtype=torch.int32, device="cuda")
    assert lib.decode_batch(out.data_ptr(), frames, cap, used.data_ptr(), 0, 4, back.data_ptr(), n, bused.data_ptr(),
                            fmts.data_ptr(), res.data_ptr()) == 0
    assert res.tolist() == [0] * frames and bused.tolist() == [n] * frames and fmts.tolist() == [YCOCG] * frames
    assert torch.equal(back, tex)
    # max_chunks too small is reported per frame, not a crash
    assert lib.decode_batch(out.data_ptr(), frames, cap, used.data_ptr(), 0, 2, back.data_ptr(), n, bused.data_ptr(),
                            fmts.data_ptr(), res.data_ptr()) == 0
    assert res.tolist() == [1] * frames


@pytest.mark.parametrize("w,h,codec_name,k", [(1920, 1080, "Hap1", 1), (3840, 2160, "Hap1", 1), (3840, 2160, "HapY", 8),
                                               (7680, 4320, "HapM", 32)])
def test_full_size_roundtrip_properties(lib, w, h, codec_name, k):
    """BASELINE.json configs 1-4 at full size: encode on the GPU, decode on the GPU AND in the reference
    (bit-exact texture bytes), decoded picture close to the source."""
    import hap_b200.lib as L
    codec = getattr(L, "HapB200Codec_" + codec_name)
    img = synth.frame(w, h, 0, alpha="ramp" if codec_name == "HapM" else "opaque", device="cuda")
    cap = (lib.max_encoded_length_rgba(w, h, codec, k) + 15) // 16 * 16
    out = torch.zeros(cap, dtype=torch.uint8, device="cuda")
    used = torch.zeros(1, dtype=torch.int64, device="cuda")
    assert lib.encode_rgba_batch(img.data_ptr(), 1, img.numel(), w, h, codec, 1, k, out.data_ptr(), cap, used.data_ptr()) == 0
    frame = out[: int(used[0])].cpu().numpy().tobytes()
    ref = oracles.ref_abi() or oracles.oracle_abi()
    ntex = 2 if codec_name == "HapM" else 1
    assert lib.texture_count(frame) == (0, ntex)
    for i in range(ntex):
        n = lib.texture_bytes(w, h, codec, i)
        a = ref.decode(frame, i, n)
        b = lib.decode(frame, i, n)
        assert a[0] == 0 and b[0] == 0 and a[1] == b[1] and a[2] == b[2] and len(a[1]) == n
    r, rgba = lib.decode_rgba(frame, w, h)
    assert r == 0
    dec = np.frombuffer(rgba, np.uint8).reshape(h, w, 4)
    src = img.cpu().numpy()
    ch = (0, 1, 2, 3) if codec_name == "HapM" else (0, 1, 2)
    assert oracles.psnr(src, dec, ch) > 38.0


def test_decode_rgba_batch_matches_oracle_block_decoder(lib):
    """Frames -> RGBA in one batched call (Snappy decode + block decode + YCoCg / alpha merge on the GPU)
    equals the oracle's block decoder applied to the reference-decoded texture bytes."""
    import hap_b200.lib as L
    w, h, frames, k = 256, 128, 5, 4
    for codec_name, kinds in (("HapY", ["ycocg"]), ("HapM", ["ycocg", "bc4"]), ("Hap1", ["bc1"]), ("Hap5", ["bc3"])):
        codec = getattr(L, "HapB200Codec_" + codec_name)
        imgs = torch.stack([synth.frame(w, h, i, alpha="ramp", device="cuda") for i in range(frames)])
        cap = (lib.max_encoded_length_rgba(w, h, codec, k) + 15) // 16 * 16
        out = torch.zeros(frames * cap, dtype=torch.uint8, device="cuda")
        used = torch.zeros(frames, dtype=torch.int64, device="cuda")
        assert lib.encode_rgba_batch(imgs.data_ptr(), frames, w * h * 4, w, h, codec, 1, k, out.data_ptr(), cap, used.data_ptr()) == 0
        rgba = torch.zeros((frames, h, w, 4), dtype=torch.uint8, device="cuda")
        res = torch.full((frames,), 9, dtype=torch.int32, device="cuda")
        assert lib.decode_rgba_batch(out.data_ptr(), frames, cap, used.data_ptr(), k, codec, w, h, rgba.data_ptr(), w * h * 4,
                                     res.data_ptr()) == 0
        assert res.tolist() == [0] * frames
        ref = oracles.ref_abi() or oracles.oracle_abi()
        host = out.cpu().numpy()
        for f in range(frames):
            fr = host[f * cap: f * cap + int(used[f])].tobytes()
            t0 = ref.decode(fr, 0, lib.texture_bytes(w, h, codec, 0))[1]
            want = oracles.bc_decode(kinds[0], t0, w, h)
            if kinds[0] == "bc4":
                want = np.stack([want, want, want, np.full_like(want, 255)], -1)
            if len(kinds) == 2:
                t1 = ref.decode(fr, 1, lib.texture_bytes(w, h, codec, 1))[1]
                want = want.copy()
                want[..., 3] = oracles.bc_decode("bc4", t1, w, h)
            assert np.array_equal(rgba[f].cpu().numpy(), want), (codec_name, f)
        # a frame of another flavour is reported per frame, not decoded
        other = L.HapB200Codec_Hap1 if codec_name != "Hap1" else L.HapB200Codec_HapY
        assert lib.decode_rgba_batch(out.data_ptr(), frames, cap, used.data_ptr(), k, other, w, h, rgba.data_ptr(), w * h * 4,
                                     res.data_ptr()) == 0
        assert all(r in (2, 3) for r in res.tolist())  # wrong size for the claimed flavour, or wrong format


def test_16k_frame_roundtrip(lib):
    """BASELINE.json config 5's frame size: one 16384 x 16384 RGBA frame (1 GiB) -> Hap Q, 64 chunks -> decoded on
    the GPU; the decoded texture must equal the block encoder's output (kept on the device, 256 MiB)."""
    import hap_b200.lib as L
    w = h = 16384
    codec, k = L.HapB200Codec_HapY, 64
    free, _ = torch.cuda.mem_get_info()
    if free < 6 * 2 ** 30:
        pytest.skip("not enough free device memory")
    img = torch.empty((h, w, 4), dtype=torch.uint8, device="cuda")
    tile = synth.frame(2048, 2048, 0, device="cuda")
    for y in range(0, h, 2048):
        for x in range(0, w, 2048):
            img[y:y + 2048, x:x + 2048] = tile
    n = lib.texture_bytes(w, h, codec)
    blocks = torch.zeros(n, dtype=torch.uint8, device="cuda")
    assert lib.block_encode_batch(img.data_ptr(), 1, img.numel(), w, h, codec, blocks.data_ptr(), n) == 0
    cap = (lib.max_encoded_length_rgba(w, h, codec, k) + 15) // 16 * 16
    out = torch.zeros(cap, dtype=torch.uint8, device="cuda")
    used = torch.zeros(1, dtype=torch.int64, device="cuda")
    assert lib.encode_rgba_batch(img.data_ptr(), 1, img.numel(), w, h, codec, 1, k, out.data_ptr(), cap, used.data_ptr()) == 0
    nbytes = int(used[0])
    assert out[:4].tolist() == [0, 0, 0, 0xCF]          # 8-byte header, complex, YCoCg
    assert nbytes < n
    back = torch.zeros(n, dtype=torch.uint8, device="cuda")
    bused = torch.zeros(1, dtype=torch.int64, device="cuda")
    fmts = torch.zeros(1, dtype=torch.int32, device="cuda")
    res = torch.full((1,), 9, dtype=torch.int32, device="cuda")
    assert lib.decode_batch(out.data_ptr(), 1, cap, used.data_ptr(), 0, k, back.data_ptr(), n, bused.data_ptr(), fmts.data_ptr(),
                            res.data_ptr()) == 0
    assert res.tolist() == [0] and bused.tolist() == [n] and fmts.tolist() == [1]
    assert torch.equal(back, blocks)
    # the host-side header walk agrees (chunk count as the reference limits it)
    head = out[: 4096].cpu().numpy().tobytes()
    assert head[8:12] == (5 * 64 + 8).to_bytes(3, "little") + b"\x01"


def test_concurrent_host_calls_are_reentrant(lib):
    """The reference is re-entrant (no globals in hap.c); so are the host-pointer entry points here: calls from
    many host threads run on pooled streams at the same time and must not mix their buffers."""
    from concurrent.futures import ThreadPoolExecutor
    rng = np.random.default_rng(21)
    payloads = [dxt_like(rng, int(rng.integers(2000, 9000)), 16) for _ in range(24)]
    orc = oracles.oracle_abi()

    def work(i):
        p = payloads[i]
        k = 1 + i % 7
        r, f = lib.encode([p], [YCOCG], [HapCompressorSnappy], [k])
        assert r == 0
        r2, back, fmt, calls = lib.decode(f, 0, len(p))
        return r2 == 0 and back == p and fmt == YCOCG and orc.decode(f, 0, len(p))[1] == p

    with ThreadPoolExecutor(8) as pool:
        assert all(pool.map(work, range(len(payloads))))


def test_banded_single_frame_encode_assembles_to_one_frame(lib):
    """SURVEY.md 8e, second case, on one GPU: a picture cut into three bands of block rows, each band encoded on its own
    (as each rank would), the band frames spliced by sharding.assemble_banded_frame; the result decodes here and in
    the oracle to the bands' textures one after the other, with the bands' chunk counts added up."""
    import hap_b200.lib as L
    from hap_b200 import sharding
    w, h = 512, 384
    img = synth.frame(w, h, 5).numpy()
    rows = [(0, 128), (128, 256), (256, 384)]
    ks = [2, 1, 3]
    band_frames, band_tex = [], []
    for (y0, y1), k in zip(rows, ks):
        band = np.ascontiguousarray(img[y0:y1])
        r, f = lib.encode_rgba(band, w, y1 - y0, L.HapB200Codec_HapY, hap_b200.HapCompressorSnappy, k)
        assert r == 0
        n = lib.texture_bytes(w, y1 - y0, L.HapB200Codec_HapY)
        r, tex, fmt, _ = lib.decode(f, 0, n)
        assert r == 0 and fmt == hap_b200.HapTextureFormat_YCoCg_DXT5
        band_frames.append(f)
        band_tex.append(tex)
    whole = sharding.assemble_banded_frame(band_frames)
    want = b"".join(band_tex)
    assert lib.chunk_count(whole, 0) == (0, sum(lib.chunk_count(f, 0)[1] for f in band_frames))
    r, tex, fmt, calls = lib.decode(whole, 0, len(want))
    assert r == 0 and tex == want and fmt == hap_b200.HapTextureFormat_YCoCg_DXT5
    ro, tex_o, _, _ = oracles.oracle_abi().decode(whole, 0, len(want))
    assert ro == 0 and tex_o == want
    # and the whole picture's texture is the same blocks: bands are whole block rows
    r, f_all = lib.encode_rgba(img, w, h, L.HapB200Codec_HapY, hap_b200.HapCompressorSnappy, 6)
    r2, tex_all, _, _ = lib.decode(f_all, 0, len(want))
    assert r == 0 and r2 == 0 and tex_all == want


def test_rgba_batch_texture_cannot_overrun_its_share_of_the_slot(lib):
    """ADVICE r1 (high): in HapB200DecodeRGBABatch both textures of a Hap Q Alpha frame share one scratch slot.  A
    hostile frame whose ALPHA texture declares more bytes than an RGTC1 plane has (but no more than the slot is wide)
    used to pass the size check and write over the next frame's colour texture.  It must be refused per frame, and the
    neighbouring frame must decode to the same picture as when it is decoded alone."""
    import hap_b200.lib as L
    w, h, k = 128, 64, 2
    codec = L.HapB200Codec_HapM
    img = synth.frame(w, h, 0, alpha="ramp", device="cuda")
    cap = (lib.max_encoded_length_rgba(w, h, codec, k) + 15) // 16 * 16
    one = torch.zeros(cap, dtype=torch.uint8, device="cuda")
    used1 = torch.zeros(1, dtype=torch.int64, device="cuda")
    assert lib.encode_rgba_batch(img.data_ptr(), 1, img.numel(), w, h, codec, 1, k, one.data_ptr(), cap, used1.data_ptr()) == 0
    good = one[: int(used1[0])].cpu().numpy().tobytes()
    t0, t1 = lib.texture_bytes(w, h, codec, 0), lib.texture_bytes(w, h, codec, 1)
    r, tex0, _, _ = lib.decode(good, 0, t0)
    assert r == 0
    # hostile twin: same colour section, alpha section = a verbatim (0xA1) section of t0 + t1 - 16 bytes
    fat = bytes([0x77]) * (t0 + t1 - 16)
    r, sec0 = lib.encode([tex0], [YCOCG], [0], [1])
    assert r == 0
    sec1 = len(fat).to_bytes(3, "little") + bytes([0xA1]) + fat
    body = sec0 + sec1
    hostile = len(body).to_bytes(3, "little") + bytes([0x0D]) + body
    assert lib.texture_count(hostile) == (0, 2) and lib.texture_format(hostile, 1) == (0, RGTC1)
    big = max(cap, (len(hostile) + 15) // 16 * 16)
    buf = torch.zeros(2 * big, dtype=torch.uint8, device="cuda")
    buf[: len(hostile)] = torch.frombuffer(bytearray(hostile), dtype=torch.uint8).cuda()
    buf[big: big + len(good)] = torch.frombuffer(bytearray(good), dtype=torch.uint8).cuda()
    used = torch.tensor([len(hostile), len(good)], dtype=torch.int64, device="cuda")
    rgba = torch.full((2, h, w, 4), 0xEE, dtype=torch.uint8, device="cuda")
    res = torch.full((2,), 9, dtype=torch.int32, device="cuda")
    assert lib.decode_rgba_batch(buf.data_ptr(), 2, big, used.data_ptr(), k, codec, w, h, rgba.data_ptr(), w * h * 4, res.data_ptr()) == 0
    assert res.tolist()[0] in (2, 3) and res.tolist()[1] == 0, res.tolist()
    alone = torch.zeros((1, h, w, 4), dtype=torch.uint8, device="cuda")
    r1 = torch.full((1,), 9, dtype=torch.int32, device="cuda")
    assert lib.decode_rgba_batch(one.data_ptr(), 1, cap, used1.data_ptr(), k, codec, w, h, alone.data_ptr(), w * h * 4, r1.data_ptr()) == 0
    assert r1.tolist() == [0] and torch.equal(rgba[1], alone[0])
    assert int(rgba[0].max()) == 0          # the refused frame's picture is zeros, not recycled scratch


@pytest.fixture
def index_on(lib):
    lib.set_option(lib.OPTION_WRITE_INDEX, 1)
    yield lib
    lib.set_option(lib.OPTION_WRITE_INDEX, 0)
    lib.set_option(lib.OPTION_USE_INDEX, 1)


@pytest.mark.parametrize("w,h,codec_name,k", [(1920, 1080, "Hap1", 1), (3840, 2160, "HapY", 8), (2048, 1024, "HapM", 5), (512, 256, "Hap5", 3)])
def test_frames_with_fragment_index(index_on, w, h, codec_name, k):
    """hap_index.h: the encoder appends the fragment index behind the frame.  The frame proper is byte-identical to the frame
    written without it; the reference decodes it (ignoring the trailing section) to the texture; this decoder gives the same
    bytes with the index, without it (on-the-fly index) and when the index has been damaged (repair pass)."""
    import hap_b200.lib as L
    lib = index_on
    codec = getattr(L, "HapB200Codec_" + codec_name)
    img = synth.frame(w, h, 3, alpha="ramp" if codec_name in ("HapM", "Hap5") else "opaque", device="cuda")
    cap = (lib.max_encoded_length_rgba(w, h, codec, k) + 15) // 16 * 16
    out = torch.zeros(2 * cap, dtype=torch.uint8, device="cuda")
    used = torch.zeros(2, dtype=torch.int64, device="cuda")
    assert lib.encode_rgba_batch(img.data_ptr(), 1, img.numel(), w, h, codec, 1, k, out.data_ptr(), cap, used.data_ptr()) == 0
    lib.set_option(lib.OPTION_WRITE_INDEX, 0)
    assert lib.encode_rgba_batch(img.data_ptr(), 1, img.numel(), w, h, codec, 1, k, out.data_ptr() + cap, cap, used.data_ptr() + 8) == 0
    lib.set_option(lib.OPTION_WRITE_INDEX, 1)
    host = out.cpu().numpy()
    with_ix, plain = host[: int(used[0])].tobytes(), host[cap: cap + int(used[1])].tobytes()
    assert len(with_ix) > len(plain) and with_ix[: len(plain)] == plain
    assert with_ix[len(plain) + 3] == 0xFB and with_ix[len(plain) + 4: len(plain) + 8] == b"HB2I"
    assert len(with_ix) <= 1.02 * len(plain) + 64          # about one per cent
    ref = oracles.ref_abi() or oracles.oracle_abi()
    ntex = 2 if codec_name == "HapM" else 1
    damaged = bytearray(with_ix)
    rng = np.random.default_rng(7)
    for _ in range(6):
        damaged[len(plain) + 40 + int(rng.integers(0, len(with_ix) - len(plain) - 40))] ^= 1 << int(rng.integers(0, 8))
    for i in range(ntex):
        n = lib.texture_bytes(w, h, codec, i)
        want = ref.decode(with_ix, i, n)
        assert want[0] == 0 and len(want[1]) == n
        assert lib.decode(with_ix, i, n)[:3] == want[:3]
        assert lib.decode(bytes(damaged), i, n)[:3] == want[:3]
        lib.set_option(lib.OPTION_USE_INDEX, 0)
        assert lib.decode(with_ix, i, n)[:3] == want[:3]
        lib.set_option(lib.OPTION_USE_INDEX, 1)
    # batch path: three copies, the middle one damaged
    F = 3
    bcap = (len(with_ix) + 63) // 64 * 64
    buf = torch.zeros(F * bcap, dtype=torch.uint8, device="cuda")
    for f, fr in enumerate((with_ix, bytes(damaged), with_ix)):
        buf[f * bcap: f * bcap + len(fr)] = torch.frombuffer(bytearray(fr), dtype=torch.uint8).cuda()
    lens = torch.tensor([len(with_ix)] * F, dtype=torch.int64, device="cuda")
    for i in range(ntex):
        n = lib.texture_bytes(w, h, codec, i)
        stride = (n + 15) // 16 * 16
        tex = torch.zeros(F * stride, dtype=torch.uint8, device="cuda")
        tu = torch.zeros(F, dtype=torch.int64, device="cuda")
        tf = torch.zeros(F, dtype=torch.int32, device="cuda")
        res = torch.full((F,), 9, dtype=torch.int32, device="cuda")
        assert lib.decode_batch(buf.data_ptr(), F, bcap, lens.data_ptr(), i, k, tex.data_ptr(), stride, tu.data_ptr(), tf.data_ptr(), res.data_ptr()) == 0
        assert res.tolist() == [0] * F and tu.tolist() == [n] * F
        want = torch.frombuffer(bytearray(ref.decode(with_ix, i, n)[1]), dtype=torch.uint8).cuda()
        for f in range(F):
            assert torch.equal(tex[f * stride: f * stride + n], want), (i, f)


@pytest.mark.parametrize("with_index", [0, 1])
def test_chunk_offset_table_option(lib, with_index):
    """HAPB200_OPTION_WRITE_OFFSET_TABLE (SURVEY.md 8f4): the optional table of HapVideoDRAFT.md:126-128 is written, chunks
    start on 16-byte boundaries of the frame, gaps are zero; the reference (hap.c:800-803 honours the table) and this
    decoder give the same texture as for the packed layout."""
    import hap_b200.lib as L
    w, h, k = 1024, 512, 8
    codec = L.HapB200Codec_HapY
    img = synth.frame(w, h, 9).numpy()
    lib.set_option(lib.OPTION_WRITE_INDEX, with_index)
    try:
        r, plain = lib.encode_rgba(img, w, h, codec, 1, k)
        lib.set_option(lib.OPTION_WRITE_OFFSET_TABLE, 1)
        r2, cot = lib.encode_rgba(img, w, h, codec, 1, k)
    finally:
        lib.set_option(lib.OPTION_WRITE_OFFSET_TABLE, 0)
        lib.set_option(lib.OPTION_WRITE_INDEX, 0)
    assert r == 0 and r2 == 0 and cot != plain
    n = lib.texture_bytes(w, h, codec)
    ref = oracles.ref_abi() or oracles.oracle_abi()
    want = ref.decode(plain, 0, n)
    assert want[0] == 0
    assert ref.decode(cot, 0, n)[:3] == want[:3]
    assert lib.decode(cot, 0, n)[:3] == want[:3] and lib.chunk_count(cot, 0) == (0, k)
    # layout: DI container = compressor table, size table, offset table (9k + 12 bytes); aligned chunk starts
    di_len = int.from_bytes(cot[4:7], "little")
    assert cot[7] == 0x01 and di_len == 9 * k + 12 and cot[8 + k + 4 + 4 * k + 4 + 3] == 0x04
    data0 = 8 + di_len
    otab = 8 + 4 + k + 4 + 4 * k + 4
    sizes = [int.from_bytes(cot[8 + 4 + k + 4 + 4 * c: 8 + 4 + k + 8 + 4 * c], "little") for c in range(k)]
    offs = [int.from_bytes(cot[otab + 4 * c: otab + 4 * c + 4], "little") for c in range(k)]
    for c in range(k):
        assert (data0 + offs[c]) % 16 == 0
        if c + 1 < k:
            assert offs[c + 1] >= offs[c] + sizes[c] and set(cot[data0 + offs[c] + sizes[c]: data0 + offs[c + 1]]) <= {0}
