"""Pins the bytes the encoder writes.  The other tests only check that frames decode to their input; these compare the
SHA-256 of every encoded frame with digests recorded from an earlier build (tests/golden/encode_sha256.json), so a
change to the fragment compressor that is meant to rearrange work and not the output is checked byte for byte.

The digests were recorded with the build before the fragment compressor (K5) ran two 512-thread CTAs per SM:
    emulator:  g++ -std=c++17 -O1 -w -I hap_b200/csrc -I tests/emu -I oracle tests/emu/encode_sha256_emu.cc \\
                   oracle/snappy_oracle.c oracle/hap_oracle.c oracle/bc_oracle.c -ldl -lm -o sha && ./sha 1
    GPU (B200): python tests/test_encode_bytes.py      (prints the "gpu" entry as JSON)
An intended change of the encoded bytes records them again the same way."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "encode_sha256.json")
BUILD = os.path.join(ROOT, "tests", "emu", "_build")
EMU_MODES = 3   # thread resume orders of the emulator: forward, reverse, seeded shuffle (each also with its own grid size)

# Seeded synth frames, 720x480, 4 chunks: every chunk is 2 or 3 fragments and its last fragment is partial
GPU_W, GPU_H, GPU_FRAMES, GPU_CHUNKS = 720, 480, 3, 4
GPU_CODECS = (("hap", 0, "opaque"), ("hap_alpha", 1, "ramp"), ("hap_q", 2, "opaque"), ("hap_q_alpha", 3, "ramp"),
              ("hap_alpha_only", 4, "ramp"))   # (name, HapB200Codec_*, synth alpha)


def golden():
    with open(GOLDEN) as f:
        return json.load(f)


def test_emulated_encoder_bytes_unchanged():
    os.makedirs(BUILD, exist_ok=True)
    exe = os.path.join(BUILD, "encode_sha256_emu")
    inc = ["-I", os.path.join(ROOT, "hap_b200", "csrc"), "-I", os.path.join(ROOT, "tests", "emu"), "-I", os.path.join(ROOT, "oracle")]
    orc = [os.path.join(ROOT, "oracle", f) for f in ("snappy_oracle.c", "hap_oracle.c", "bc_oracle.c")]
    subprocess.run(["g++", "-std=c++17", "-O1", "-w"] + inc + [os.path.join(ROOT, "tests", "emu", "encode_sha256_emu.cc")] + orc
                   + ["-ldl", "-lm", "-o", exe], check=True)
    p = subprocess.run([exe, str(EMU_MODES)], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    want = golden()["emulator"]
    got = {}
    for line in p.stdout.splitlines():
        if line.startswith("sha256 "):
            _, mode, name, digest = line.split()
            got.setdefault(name, {})[int(mode)] = digest
    assert sorted(got) == sorted(want)
    bad = [(name, mode) for name, per_mode in got.items() for mode, d in per_mode.items() if d != want[name]]
    assert all(len(per_mode) == EMU_MODES for per_mode in got.values())
    assert bad == []


def gpu_frame_digests():
    """{codec name: [SHA-256 of every frame]} of a seeded batch encoded on cuda:0 (Snappy, default options)."""
    import hashlib

    import torch

    import hap_b200
    from hap_b200 import synth

    lib = hap_b200.load()
    dev = torch.device("cuda", 0)
    out = {}
    for name, codec, alpha in GPU_CODECS:
        imgs = synth.frames(GPU_W, GPU_H, GPU_FRAMES, alpha=alpha).to(dev)
        cap = (lib.max_encoded_length_rgba(GPU_W, GPU_H, codec, GPU_CHUNKS) + 255) // 256 * 256
        frames = torch.zeros((GPU_FRAMES, cap), dtype=torch.uint8, device=dev)
        used = torch.zeros(GPU_FRAMES, dtype=torch.int64, device=dev)
        r = lib.encode_rgba_batch(imgs.data_ptr(), GPU_FRAMES, GPU_W * GPU_H * 4, GPU_W, GPU_H, codec, 1, GPU_CHUNKS,
                                  frames.data_ptr(), cap, used.data_ptr())
        assert r == 0, (name, r)
        host = frames.cpu().numpy()
        out[name] = [hashlib.sha256(host[f, : int(used[f])].tobytes()).hexdigest() for f in range(GPU_FRAMES)]
    return out


@pytest.mark.gpu
def test_gpu_encoder_bytes_unchanged():
    assert gpu_frame_digests() == golden()["gpu"]


if __name__ == "__main__":
    sys.path.insert(0, ROOT)
    print(json.dumps(gpu_frame_digests(), indent=1))
