"""QuickTime container layer (include/hap_mov.h, SURVEY.md 8(f) rank 1): the writer's files are read back
bit-exactly by our reader AND by FFmpeg's mov demuxer (through OpenCV, an independent implementation); the reader
reads movies laid out by an independent writer (a few lines of struct.pack below) in the layouts other tools
produce, and refuses damaged files.  Host code only: runs without a GPU."""
import os
import struct

import numpy as np
import pytest

import hap_b200
from hap_b200 import mov
from hap_b200.abi import (HapCompressorNone, HapTextureFormat_A_RGTC1, HapTextureFormat_RGB_DXT1,
                          HapTextureFormat_RGBA_DXT5, HapTextureFormat_YCoCg_DXT5)


@pytest.fixture(scope="module")
def lib():
    from hap_b200 import build
    build.build()
    return hap_b200.load()


def hap_frames(lib, w, h, n, fmt=HapTextureFormat_RGB_DXT1, seed=0):
    """n valid Hap frames (verbatim sections: host-only encode path) of different sizes"""
    rng = np.random.default_rng(seed)
    per = 8 if fmt in (HapTextureFormat_RGB_DXT1, HapTextureFormat_A_RGTC1) else 16
    out = []
    for i in range(n):
        tex = rng.integers(0, 256, (w // 4) * (h // 4) * per, dtype=np.uint8).tobytes()
        r, f = lib.encode([tex], [fmt], [HapCompressorNone], [1])
        assert r == 0
        out.append(f)
    return out


def test_fourcc_names(lib):
    w, h = 16, 8
    for fmt, name in ((HapTextureFormat_RGB_DXT1, "Hap1"), (HapTextureFormat_RGBA_DXT5, "Hap5"), (HapTextureFormat_YCoCg_DXT5, "HapY"),
                      (HapTextureFormat_A_RGTC1, "HapA")):
        assert mov.fourcc_for_frame(hap_frames(lib, w, h, 1, fmt)[0]) == (0, name)
    y = bytes((w // 4) * (h // 4) * 16)
    a = bytes((w // 4) * (h // 4) * 8)
    r, f = lib.encode([y, a], [HapTextureFormat_YCoCg_DXT5, HapTextureFormat_A_RGTC1], [HapCompressorNone] * 2, [1, 1])
    assert r == 0 and mov.fourcc_for_frame(f) == (0, "HapM")
    assert mov.fourcc_for_frame(b"\x00\x01\x02")[0] != 0


def test_write_then_read_back(lib, tmp_path):
    frames = hap_frames(lib, 64, 32, 7)
    path = str(tmp_path / "a.mov")
    ticks = [100, 100, 100, 250, 250, 100, 40]
    with mov.MovWriter(path, "Hap1", 64, 32, 3000) as wr:
        for f, t in zip(frames, ticks):
            assert wr.write(f, t) == 0
        assert wr.write(b"", 1) != 0          # empty samples are refused
    with mov.MovReader(path) as rd:
        assert (rd.fourcc, rd.width, rd.height, rd.frames, rd.timescale, rd.duration) == ("Hap1", 64, 32, 7, 3000, sum(ticks))
        for i, (f, t) in enumerate(zip(frames, ticks)):
            assert rd.read(i) == (0, f, t)
        assert rd.read(7)[0] == 1 and rd.frame_bytes(7) == 0          # Bad_Arguments past the end
        assert rd.read(0, capacity=10)[0] == 2                        # Buffer_Too_Small


def test_ffmpeg_demuxes_our_movie(lib, tmp_path):
    """FFmpeg's QuickTime demuxer (via OpenCV) is the independent reader of what our writer produced."""
    cv2 = pytest.importorskip("cv2")
    frames = hap_frames(lib, 128, 64, 5, HapTextureFormat_YCoCg_DXT5)
    path = str(tmp_path / "q.mov")
    with mov.MovWriter(path, "HapY", 128, 64, 600) as wr:
        for f in frames:
            assert wr.write(f, 20) == 0
    cap = cv2.VideoCapture(path, cv2.CAP_FFMPEG)
    if not cap.isOpened():
        pytest.skip("this OpenCV build cannot open QuickTime files")
    try:
        assert int(cap.get(cv2.CAP_PROP_FRAME_WIDTH)) == 128 and int(cap.get(cv2.CAP_PROP_FRAME_HEIGHT)) == 64
        assert int(cap.get(cv2.CAP_PROP_FRAME_COUNT)) == 5
        assert abs(cap.get(cv2.CAP_PROP_FPS) - 30.0) < 1e-6
        cc = int(cap.get(cv2.CAP_PROP_FOURCC))
        # FFmpeg files every Hap flavour under one codec id; OpenCV reports that id's first tag ('Hap1') or the file's own
        assert struct.pack("<I", cc) in (b"HapY", b"Hap1")
        # raw packets, when this build hands them out: byte-identical samples
        if cap.set(cv2.CAP_PROP_FORMAT, -1):
            got = []
            while True:
                ok, pkt = cap.read()
                if not ok:
                    break
                got.append(np.asarray(pkt).tobytes())
            if got:
                assert got == frames
    finally:
        cap.release()


# ---- an independent writer: the layouts other tools produce ---------------------------------------------------

def atom(t, body):
    return struct.pack(">I4s", 8 + len(body), t) + body


def atom64(t, body):
    return struct.pack(">I4sQ", 1, t, 16 + len(body)) + body


def build_movie(frames, codec=b"Hap5", w=32, h=16, samples_per_chunk=3, co64=False, mdat64=False, moov_first=False, v1=False,
                extra_track=False):
    ftyp = atom(b"ftyp", b"qt  " + struct.pack(">I", 0) + b"qt  ")
    free = atom(b"free", b"\0" * 11)

    def stbl_for(chunk_offsets):
        sd = struct.pack(">I4s6xH", 86, codec, 1) + struct.pack(">HH4sIIHHIIIH", 0, 0, b"test", 0, 512, w, h, 0x480000, 0x480000, 0, 1) + \
            bytes([3]) + b"Hap" + b"\0" * 28 + struct.pack(">Hh", 32, -1)
        assert len(sd) == 86
        stsd = atom(b"stsd", struct.pack(">II", 0, 1) + sd)
        stts = atom(b"stts", struct.pack(">II", 0, 1) + struct.pack(">II", len(frames), 10))
        nfull, rem = divmod(len(frames), samples_per_chunk)
        runs = [(1, samples_per_chunk, 1)] if nfull else []
        if rem:
            runs.append((nfull + 1, rem, 1))
        stsc = atom(b"stsc", struct.pack(">II", 0, len(runs)) + b"".join(struct.pack(">III", *r) for r in runs))
        stsz = atom(b"stsz", struct.pack(">III", 0, 0, len(frames)) + b"".join(struct.pack(">I", len(f)) for f in frames))
        if co64:
            stco = atom(b"co64", struct.pack(">II", 0, len(chunk_offsets)) + b"".join(struct.pack(">Q", o) for o in chunk_offsets))
        else:
            stco = atom(b"stco", struct.pack(">II", 0, len(chunk_offsets)) + b"".join(struct.pack(">I", o) for o in chunk_offsets))
        return atom(b"stbl", atom(b"unkn", b"xyz") + stsz + stsc + stco + stts + stsd)   # unusual order on purpose

    def moov_for(chunk_offsets):
        if v1:
            mdhd = atom(b"mdhd", struct.pack(">IQQIQHH", 1 << 24, 0, 0, 600, 10 * len(frames), 0, 0))
        else:
            mdhd = atom(b"mdhd", struct.pack(">IIIIIHH", 0, 0, 0, 600, 10 * len(frames), 0, 0))
        hdlr = atom(b"hdlr", struct.pack(">I4s4sIII", 0, b"mhlr", b"vide", 0, 0, 0) + b"\0")
        minf = atom(b"minf", atom(b"vmhd", struct.pack(">IHHHH", 1, 0x40, 0x8000, 0x8000, 0x8000)) + stbl_for(chunk_offsets))
        trak = atom(b"trak", atom(b"tkhd", b"\0" * 84) + atom(b"mdia", mdhd + hdlr + minf))
        sound = b""
        if extra_track:  # a sound track before the video track: must be skipped
            shdlr = atom(b"hdlr", struct.pack(">I4s4sIII", 0, b"mhlr", b"soun", 0, 0, 0) + b"\0")
            sound = atom(b"trak", atom(b"tkhd", b"\0" * 84) + atom(b"mdia", mdhd + shdlr + atom(b"minf", b"")))
        return atom(b"moov", atom(b"mvhd", b"\0" * 100) + sound + trak)

    def layout(data_start):
        offs, pos, chunk_offsets = [], data_start, []
        for i, f in enumerate(frames):
            if i % samples_per_chunk == 0:
                chunk_offsets.append(pos)
            offs.append(pos)
            pos += len(f)
        return chunk_offsets

    payload = b"".join(frames)
    mdat = (atom64 if mdat64 else atom)(b"mdat", payload)
    mdat_hdr = 16 if mdat64 else 8
    if moov_first:
        size_moov = len(moov_for([0] * ((len(frames) + samples_per_chunk - 1) // samples_per_chunk)))
        start = len(ftyp) + size_moov + len(free) + mdat_hdr
        return ftyp + moov_for(layout(start)) + free + mdat
    start = len(ftyp) + len(free) + mdat_hdr
    return ftyp + free + mdat + moov_for(layout(start))


@pytest.mark.parametrize("kw", [dict(), dict(samples_per_chunk=1), dict(co64=True, mdat64=True), dict(moov_first=True, samples_per_chunk=2),
                                dict(v1=True, extra_track=True, samples_per_chunk=5)])
def test_reader_on_independently_built_movies(lib, tmp_path, kw):
    frames = hap_frames(lib, 32, 16, 8, HapTextureFormat_RGBA_DXT5, seed=3)
    frames = [f + bytes(i) for i, f in enumerate(frames)]      # different sizes (trailing bytes belong to the sample)
    path = str(tmp_path / "ind.mov")
    open(path, "wb").write(build_movie(frames, **kw))
    with mov.MovReader(path) as rd:
        assert (rd.fourcc, rd.width, rd.height, rd.frames, rd.timescale) == ("Hap5", 32, 16, 8, 600)
        for i, f in enumerate(frames):
            assert rd.read(i) == (0, f, 10)


def test_reader_refuses_damaged_and_foreign_files(lib, tmp_path):
    frames = hap_frames(lib, 32, 16, 4, HapTextureFormat_RGBA_DXT5)
    good = build_movie(frames)
    p = str(tmp_path / "x.mov")

    def opens(data):
        open(p, "wb").write(data)
        try:
            mov.MovReader(p).close()
            return True
        except ValueError:
            return False

    assert opens(good)
    assert not opens(b"")
    assert not opens(good[: len(good) // 2])                    # moov cut off
    assert not opens(good.replace(b"Hap5", b"avc1"))            # not a Hap track
    assert not opens(build_movie(frames, codec=b"Hap5")[:-40])  # truncated inside the sample tables
    # sample table pointing outside the file
    bad = bytearray(good)
    i = bad.rfind(b"stco")
    bad[i + 12: i + 16] = struct.pack(">I", 0x7FFFFFF0)
    assert not opens(bytes(bad))
    # an atom that claims to be larger than its parent
    bad = bytearray(good)
    i = bad.rfind(b"stbl")
    bad[i - 4: i] = struct.pack(">I", 0x10000000)
    assert not opens(bytes(bad))
    with pytest.raises(ValueError):
        mov.MovReader(str(tmp_path / "missing.mov"))
    with pytest.raises(ValueError):
        mov.MovWriter(str(tmp_path / "w.mov"), "avc1", 16, 16, 600)


def test_ffmpeg_decodes_our_frames(lib, tmp_path):
    """FFmpeg's own Hap decoder (libavcodec hapdec + texturedsp, reached through OpenCV) decodes the frames of our
    movie to the picture our block decoder oracle gets from the same texture, to within its rounding."""
    cv2 = pytest.importorskip("cv2")
    import oracles
    import twin
    from hap_b200 import synth
    w, h = 256, 128
    img = synth.frame(w, h, 0).numpy()
    for kind, fmt, cc in (("bc1", HapTextureFormat_RGB_DXT1, "Hap1"), ("bc3", HapTextureFormat_RGBA_DXT5, "Hap5"),
                          ("ycocg", HapTextureFormat_YCoCg_DXT5, "HapY")):
        tex = twin.encode(kind, img)
        r, f = lib.encode([tex], [fmt], [HapCompressorNone], [1])
        assert r == 0
        path = str(tmp_path / f"{cc}.mov")
        with mov.MovWriter(path, cc, w, h, 600) as wr:
            for _ in range(2):
                assert wr.write(f, 20) == 0
        cap = cv2.VideoCapture(path, cv2.CAP_FFMPEG)
        ok, bgr = cap.read() if cap.isOpened() else (False, None)
        cap.release()
        if not ok:
            pytest.skip("this OpenCV/FFmpeg build has no Hap decoder")
        ref = oracles.bc_decode(kind, tex, w, h)[..., :3][..., ::-1]
        assert np.abs(bgr.astype(int) - ref.astype(int)).max() <= 3, cc


def test_reader_survives_damaged_movies_under_sanitizers(tmp_path):
    """tests/emu/test_mov_fuzz.cc: the reader source under ASan + UBSan on 3000 truncated / bit-flipped / spliced
    movies -- it refuses them or hands out frames that lie inside the file."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "mov_fuzz")
    subprocess.run(["g++", "-std=c++17", "-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined",
                    "-I", os.path.join(root, "hap_b200", "csrc"), "-I", os.path.join(root, "include"),
                    os.path.join(root, "tests", "emu", "test_mov_fuzz.cc"), "-o", exe], check=True)
    p = subprocess.run([exe, "3000"], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, ASAN_OPTIONS="detect_leaks=0"))
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-4000:]
    assert "without a fault" in p.stdout


@pytest.mark.parametrize("who", ["oracle", "reference"])
def test_ffmpeg_decodes_snappy_frames_of_oracle_and_reference(lib, tmp_path, who):
    """Closes the triangle on the CPU: Snappy-compressed, chunked frames written by the oracle port and by the
    unmodified reference build (stored in tests/golden) go through our movie writer and are decoded by FFmpeg's independent
    Hap decoder to the picture the oracle's block decoder gets from the same texture."""
    cv2 = pytest.importorskip("cv2")
    import oracles
    import twin
    from golden_util import golden, sha, unpack_frame
    from hap_b200 import synth
    from hap_b200.abi import HapCompressorSnappy
    orc = oracles.oracle_abi()
    w, h = 256, 128
    img = synth.frame(w, h, 1).numpy()
    for kind, fmt, cc, chunks in (("bc1", HapTextureFormat_RGB_DXT1, "Hap1", 1), ("ycocg", HapTextureFormat_YCoCg_DXT5, "HapY", 4)):
        if who == "oracle":
            tex = twin.encode(kind, img)
            r, f = orc.encode([tex], [fmt], [HapCompressorSnappy], [chunks])
        else:
            G = golden()["mov_frames"][kind]
            f = unpack_frame(G["frame"])
            r, tex, _, _ = orc.decode(f, 0, (w // 4) * (h // 4) * (8 if kind == "bc1" else 16))
            assert sha(tex) == G["payload_sha256"]
        assert r == 0 and mov.fourcc_for_frame(f) == (0, cc)
        path = str(tmp_path / f"{who}_{cc}.mov")
        with mov.MovWriter(path, cc, w, h, 600) as wr:
            assert wr.write(f, 20) == 0 and wr.write(f, 20) == 0
        cap = cv2.VideoCapture(path, cv2.CAP_FFMPEG)
        ok, bgr = cap.read() if cap.isOpened() else (False, None)
        cap.release()
        if not ok:
            pytest.skip("this OpenCV/FFmpeg build has no Hap decoder")
        ref = oracles.bc_decode(kind, tex, w, h)[..., :3][..., ::-1]
        assert np.abs(bgr.astype(int) - ref.astype(int)).max() <= 3, (who, cc)


def with_private_section(frame: bytes, body: bytes, typ: int = 0xFB) -> bytes:
    """Insert an unknown section behind the size table of the Decode Instructions container of a single-texture Complex
    frame with 4-byte headers: legal by hap.c:701-704, but NOT what the fragment index does (FFmpeg cannot take it)."""
    top_len = int.from_bytes(frame[0:3], "little")
    assert top_len != 0 and (frame[3] >> 4) == 0xC and frame[7] == 0x01
    di_len = int.from_bytes(frame[4:7], "little")
    extra = len(body).to_bytes(3, "little") + bytes([typ]) + body
    di_end = 8 + di_len
    out = bytearray()
    out += (top_len + len(extra)).to_bytes(3, "little") + frame[3:4]
    out += (di_len + len(extra)).to_bytes(3, "little") + frame[7:8]
    out += frame[8:di_end] + extra + frame[di_end:]
    return bytes(out)


def with_trailing_section(frame: bytes, body: bytes, typ: int = 0xFB) -> bytes:
    """A further top-level section behind the frame: where the fragment index of hap_b200/csrc/hap_index.h travels."""
    return frame + len(body).to_bytes(3, "little") + bytes([typ]) + body


def test_a_trailing_section_is_ignored_by_every_decoder(lib, tmp_path):
    """The fragment index is appended to the frame as one more top-level section.  The reference (and its port) work
    inside the first section's stated length; FFmpeg's Hap decoder does the same -- frames with and without the trailing
    section decode to the same picture, one and two textures.  (An unknown section INSIDE the Decode Instructions container,
    which hap.c:701-704 skips, is accepted by the reference but not by FFmpeg: also checked, it is why the index trails.)"""
    cv2 = pytest.importorskip("cv2")
    import oracles
    import twin
    from hap_b200 import synth
    from hap_b200.abi import HapCompressorSnappy, HapTextureFormat_A_RGTC1
    w, h = 256, 128
    img = synth.frame(w, h, 2, alpha="ramp").numpy()
    tex, alpha = twin.encode("ycocg", img), twin.encode("bc4", img)
    orc, ref = oracles.oracle_abi(), oracles.ref_abi()
    body = b"HB2I" + bytes(range(60))
    for cc, texs, fmts, chunks in (("HapY", [tex], [HapTextureFormat_YCoCg_DXT5], [4]),
                                   ("HapM", [tex, alpha], [HapTextureFormat_YCoCg_DXT5, HapTextureFormat_A_RGTC1], [4, 2])):
        r, f = orc.encode(texs, fmts, [HapCompressorSnappy] * len(texs), chunks)
        assert r == 0
        g = with_trailing_section(f, body)
        for dec in (orc, ref, lib):
            if dec is None:
                continue
            assert dec.texture_count(g) == (0, len(texs))
            for i in range(len(texs)):
                assert dec.chunk_count(g, i) == (0, chunks[i]) and dec.texture_format(g, i) == (0, fmts[i])
                if dec is not lib:   # (the library's decode needs the GPU: tests/test_gpu_parity.py)
                    assert dec.decode(g, i, len(texs[i]))[:3] == (0, texs[i], fmts[i])
        path = str(tmp_path / f"trailing_{cc}.mov")
        with mov.MovWriter(path, cc, w, h, 600) as wr:
            assert wr.write(g, 20) == 0 and wr.write(f, 20) == 0
        cap = cv2.VideoCapture(path, cv2.CAP_FFMPEG)
        ok, bgr = cap.read() if cap.isOpened() else (False, None)
        ok2, bgr2 = cap.read() if ok else (False, None)
        cap.release()
        if not ok:
            pytest.skip("this OpenCV/FFmpeg build has no Hap decoder")
        assert ok2 and np.array_equal(bgr, bgr2), cc
        refpic = oracles.bc_decode("ycocg", tex, w, h)[..., :3][..., ::-1]
        assert np.abs(bgr.astype(int) - refpic.astype(int)).max() <= 3
    # inside the Decode Instructions container: fine for hap.c, fatal for FFmpeg
    r, f = orc.encode([tex], [HapTextureFormat_YCoCg_DXT5], [HapCompressorSnappy], [4])
    inside = with_private_section(f, body)
    for dec in (orc, ref):
        if dec is not None:
            assert dec.decode(inside, 0, len(tex))[:3] == (0, tex, HapTextureFormat_YCoCg_DXT5)
    assert lib.chunk_count(inside, 0) == (0, 4)
