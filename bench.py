#!/usr/bin/env python3
"""bench.py -- Hap frame encode/decode throughput of libhap_b200.so (contract: see the task brief).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload 4k_hapq|16k_stream] [--dump-outputs DIR]

Headline workload (BASELINE.json `metric` "4K Hap-Q encode/decode GB/s per GPU", configs[2]): 3840x2160 RGBA8
synthetic video frames -> Hap Q (scaled-YCoCg-DXT5, Snappy, 8 chunks) -> decoded back to the DXT texture bytes
(what HapDecode returns).  One STEP = one pass of that round trip over a batch of `--frames` device-resident
frames per GPU (default 444 = 14.7 GB of RGBA, far larger than the 126 MB L2).  `value` = RGBA bytes pushed through
the round trip per second, all GPUs together (frames are independent: ranks take disjoint frames, weak scaling).

Legs outside the timed region (rank 0 / N=1 unless noted):
  e2e            the SAME call the reference arm times -- HapEncode + HapDecode on DXT textures in HOST memory
                 (pinned), one frame per call, host<->device copies inside the timed region (all ranks)
  e2e_rgba       HapB200EncodeRGBA + HapDecode with host RGBA (the RGBA side the reference does not have)
  roofline       per-stage CUDA-event timing of the headline step, dominant kernel vs the measured HBM peak
  extra.configs  encode-only and decode-only GB/s, fps and roofline fraction for every configuration of
                 BASELINE.json (1080p Hap x1, 4K Hap x1, 4K Hap Q x8, 8K Hap Q Alpha x32, 16K Hap Q x64)
  cpu_baseline   the reference's own CPU path on this box's host cores (see reference_cpu_path)
  extra.ref_stream_decode   decode of frames the REFERENCE encoder (hap.c + Google Snappy) made in that leg

`--impl reference` times only the reference's CPU path: unmodified hap.c (oracle/_ref) HapEncode frame-parallel over all
cores + HapDecode (frame-parallel, and through its chunk callback on a pthread pool), whole 4K Hap Q 8-chunk frames.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H, CHUNKS = 3840, 2160, int(os.environ.get("HAPB200_BENCH_CHUNKS", "8"))  # 8 = the metric's configuration (the override is for experiments)
RGBA_BYTES = 4 * W * H            # 33 177 600
DXT_BYTES = W * H                 # 8 294 400 (16 B per 4x4 block)
WORKLOAD = "hap_q_4k_rgba_encode_decode(3840x2160,YCoCg-DXT5,snappy,8chunks)"
METRIC = "hapq_4k_encode_decode_rgba_GBps"
# the workload-defining keys, identical in both arms (the driver compares the two `config` objects)
CONFIG = {"workload": WORKLOAD, "width": W, "height": H, "texture_format": "YCoCg-DXT5", "compressor": "snappy", "chunks": CHUNKS,
          "unit_of_value": "RGBA-equivalent bytes (4*W*H per frame) through HapEncode+HapDecode per second",
          "l2": "inputs larger than L2 / last-level cache"}


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured(MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback(B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region.  The sampler process is started ahead
    of the warm-up steps (nvidia-smi can take a few hundred milliseconds to print its first line, longer than a
    short timed region); every line carries nvidia-smi's own timestamp and only the lines stamped inside
    [t0, t1] -- the wall-clock interval of the timed region -- are kept."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "10"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self, t0: float = None, t1: float = None):
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.proc:
            return out
        time.sleep(0.05)   # let the line of the last interval arrive
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        inside, everything = [], []
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 8:
                    continue
                try:
                    ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                    rec = (float(f[1]), float(f[2]), [n for n, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                                                         "sw_power_cap"), f[4:8]) if v.lower().startswith("active")])
                except ValueError:
                    continue
                everything.append(rec)
                if t0 is None or (t0 - 0.005 <= ts <= t1 + 0.02):
                    inside.append(rec)
            os.unlink(self.path)
        except Exception:
            pass
        use, where = (inside, "timed region") if inside else (everything[-5:], "around the timed region (none stamped inside it)")
        if use:
            out = {"sm_mhz": statistics.median(r[0] for r in use), "sm_max_mhz": max(r[1] for r in use),
                   "reasons": sorted({n for r in use for n in r[2]}), "samples": len(use), "sampled": where}
        return out


# =====================================================================================================
# The reference's own CPU path (bounded sample): cpu_baseline and --impl reference
# =====================================================================================================

def oracle_textures(n_frames: int, cores: int):
    """YCoCg-DXT5 textures of `n_frames` synthetic 4K frames, made on the host by the oracle's block encoder (the
    reference repo ships no block compressor; these are only INPUT to the timed HapEncode).  Also returns the time one
    frame's DXT stage took on all cores (reported separately as the builder's restatement, never part of `value`)."""
    from concurrent.futures import ThreadPoolExecutor

    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracles
    from hap_b200 import synth

    pool = ThreadPoolExecutor(cores)
    rows = [(y, min(y + 16, H)) for y in range(0, H, 16)]
    out, dxt_s = [], []
    for f in range(n_frames):
        img = np.ascontiguousarray(synth.frame(W, H, f).numpy())
        t0 = time.perf_counter()
        parts = list(pool.map(lambda r: oracles.bc_encode_clusterfit("ycocg", img[r[0]:r[1]], 1), rows))
        dxt_s.append(time.perf_counter() - t0)
        out.append(np.frombuffer(b"".join(parts), dtype=np.uint8).copy())
    pool.shutdown()
    return out, statistics.median(dxt_s)


def reference_cpu_path(steps: int, warmup: int, keep_frames: int = 0):
    """One step = F whole 3840x2160 Hap Q frames (8 chunks each, Snappy) through the UNMODIFIED reference (oracle/_ref:
    hap.c + Google Snappy; the oracle port when that build is absent):
      encode  HapEncode frame-parallel over all host cores (hap.c:448-476 is serial inside a frame, no callback);
      decode  HapDecode, the faster of (a) frame-parallel over all cores, chunks serial inside a frame, and (b) one frame
              at a time with the reference's chunk callback fanned out over a pthread pool (hap.c:861) -- 8-way at most.
    DXT textures in, DXT textures out, all in host memory: exactly the reference's API boundary.  Returns a dict."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracles
    from hap_b200.abi import HapTextureFormat_YCoCg_DXT5

    cores = os.cpu_count() or 1
    drv = oracles.MtDriver()
    n_distinct = 8
    textures, dxt_stage_s = oracle_textures(n_distinct, cores)
    F = max(16, min(2 * cores, 256))
    cap = int(oracles.oracle_abi().max_encoded_length([DXT_BYTES], [HapTextureFormat_YCoCg_DXT5], [CHUNKS]))
    cap = (cap + 63) // 64 * 64
    frames = np.zeros(F * cap, np.uint8)
    back = np.zeros(F * DXT_BYTES, np.uint8)
    tex_list = [textures[i % n_distinct] for i in range(F)]
    t_enc, t_dec_fp, t_dec_cb = [], [], []
    used = None
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        r, used = drv.encode_frames(tex_list, DXT_BYTES, HapTextureFormat_YCoCg_DXT5, 1, CHUNKS, frames, cap, cores)
        t1 = time.perf_counter()
        assert r == 0, r
        r = drv.decode_frames(frames, cap, used, back, DXT_BYTES, cores)
        t2 = time.perf_counter()
        assert r == 0, r
        ncb = min(F, 16)   # callback fan-out is one frame at a time: a 16-frame sample is enough for a per-frame time
        for f in range(ncb):
            rr, n = drv.decode_one_chunk_parallel(frames.ctypes.data + f * cap, used[f], back.ctypes.data + f * DXT_BYTES, DXT_BYTES, cores)
            assert rr == 0 and n == DXT_BYTES
        t3 = time.perf_counter()
        if it >= warmup:
            t_enc.append(t1 - t0)
            t_dec_fp.append(t2 - t1)
            t_dec_cb.append((t3 - t2) / ncb * F)
    for f in (0, F - 1):
        assert (back[f * DXT_BYTES:(f + 1) * DXT_BYTES] == tex_list[f]).all(), "reference round trip is not bit-exact"
    enc, dfp, dcb = statistics.median(t_enc), statistics.median(t_dec_fp), statistics.median(t_dec_cb)
    dec = min(dfp, dcb)
    step_s = enc + dec
    res = {
        "value": F * RGBA_BYTES / step_s / 1e9, "step_s": step_s, "cores": cores, "kind": drv.kind, "frames_per_step": F,
        "encode_fps": F / enc, "decode_fps_frame_parallel": F / dfp, "decode_fps_chunk_callback": F / dcb,
        "encode_dxt_GBps": F * DXT_BYTES / enc / 1e9, "decode_dxt_GBps": F * DXT_BYTES / dec / 1e9,
        "compression_ratio": float(sum(used)) / (F * DXT_BYTES),
        "sample": (f"{F} whole 3840x2160 Hap Q frames ({CHUNKS} chunks, Snappy; {n_distinct} distinct pictures cycled) per step: "
                   f"{'unmodified reference hap.c + Google Snappy' if drv.kind == 'reference' else 'oracle port of hap.c + Snappy'} "
                   f"HapEncode frame-parallel on {cores} threads + HapDecode (best of frame-parallel / chunk-callback pool), "
                   f"host DXT in, host DXT out; median of {steps} steps"),
        # the RGBA -> DXT stage is NOT in the reference; the builder's CPU restatement of a squish-class encoder, timed
        # separately and never part of `value`
        "dxt_stage_oracle": {"what": "oracle cluster-fit YCoCg-DXT5 (1 iteration), one 4K frame on all cores -- the builder's restatement, not Vidvox/hap",
                             "s_per_frame": dxt_stage_s, "rgba_GBps": RGBA_BYTES / dxt_stage_s / 1e9,
                             "composite_rgba_GBps_with_reference": RGBA_BYTES / (dxt_stage_s + step_s / F) / 1e9},
    }
    if keep_frames:
        k = min(keep_frames, F)
        res["_frames"] = (frames[: k * cap].copy(), cap, used[:k], [tex_list[i] for i in range(k)])
    return res


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    r = reference_cpu_path(args.steps, max(args.warmup, 1))
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": r["step_s"] * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic", "config": CONFIG,
        "cpu_baseline": {"value": r["value"], "unit": "GB/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
        "e2e": {"value": r["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "detail": {k: v for k, v in r.items() if k not in ("value", "sample", "_frames")},
    }
    emit(line)


# =====================================================================================================
# GPU arm
# =====================================================================================================

class Roundtrip:
    """A device-resident batch of one configuration: RGBA frames, the encoded frames, the decoded textures."""

    def __init__(self, lib, dev, w, h, codec, chunks, frames, first_index=0, alpha="opaque"):
        import torch
        from hap_b200 import synth
        self.lib, self.dev, self.w, self.h, self.codec, self.chunks, self.F = lib, dev, w, h, codec, chunks, frames
        self.rgba_bytes = 4 * w * h
        self.rgba = torch.empty((frames, h, w, 4), dtype=torch.uint8, device=dev)
        for i in range(frames):
            self.rgba[i] = synth.frame(w, h, first_index + i, device=dev, alpha=alpha)
        self.tex_bytes = [lib.texture_bytes(w, h, codec, 0), lib.texture_bytes(w, h, codec, 1)]
        self.ntex = 2 if self.tex_bytes[1] else 1
        self.cap = (lib.max_encoded_length_rgba(w, h, codec, chunks) + 15) // 16 * 16
        self.frames = torch.empty(frames * self.cap, dtype=torch.uint8, device=dev)
        self.used = torch.zeros(frames, dtype=torch.int64, device=dev)
        self.tex = [torch.empty(frames * ((tb + 15) // 16 * 16), dtype=torch.uint8, device=dev) for tb in self.tex_bytes[: self.ntex]]
        self.tex_used = torch.zeros(frames, dtype=torch.int64, device=dev)
        self.fmts = torch.zeros(frames, dtype=torch.int32, device=dev)
        self.res = torch.zeros(frames, dtype=torch.int32, device=dev)
        # the tensors above were filled on torch's current stream; the library calls run on side streams that do not wait
        # for it (a 16K batch was encoded before its own zero-fills had landed: lengths read back as 0)
        torch.cuda.synchronize(dev)

    def encode(self, st):
        r = self.lib.encode_rgba_batch(self.rgba.data_ptr(), self.F, self.rgba_bytes, self.w, self.h, self.codec, 1, self.chunks,
                                       self.frames.data_ptr(), self.cap, self.used.data_ptr(), stream=st)
        assert r == 0, r

    def decode(self, st, frames_ptr=None, used_ptr=None):
        for ti in range(self.ntex):
            stride = (self.tex_bytes[ti] + 15) // 16 * 16
            r = self.lib.decode_batch(frames_ptr or self.frames.data_ptr(), self.F, self.cap, used_ptr or self.used.data_ptr(), ti, self.chunks,
                                      self.tex[ti].data_ptr(), stride, self.tex_used.data_ptr(), self.fmts.data_ptr(), self.res.data_ptr(), stream=st)
            assert r == 0, r

    def check(self):
        assert self.res.tolist() == [0] * self.F, f"decode failed: results {self.res.tolist()[:8]} used {self.used.tolist()[:4]} cap {self.cap}"
        assert self.tex_used.tolist() == [self.tex_bytes[self.ntex - 1]] * self.F, f"decoded sizes {self.tex_used.tolist()[:8]}"

    def mean_frame_bytes(self):
        return float(self.used.double().mean().item())


def time_on_stream(torch, stream, fn, iters, warm=2):
    with torch.cuda.stream(stream):
        for _ in range(warm):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(iters):
            fn()
        e1.record(stream)
        e1.synchronize()
    return e0.elapsed_time(e1) / iters


def extra_config_lines(lib, torch, dev, peak):
    """Encode-only and decode-only throughput of every BASELINE.json configuration (device-resident batches, CUDA events)."""
    from hap_b200.lib import HapB200Codec_Hap1, HapB200Codec_HapM, HapB200Codec_HapY
    cfgs = [("1080p_hap_dxt1_x1", 1920, 1080, HapB200Codec_Hap1, 1, 128, "opaque"),
            ("4k_hap_dxt1_x1", 3840, 2160, HapB200Codec_Hap1, 1, 48, "opaque"),
            ("4k_hapq_x8", 3840, 2160, HapB200Codec_HapY, 8, 48, "opaque"),
            ("8k_hapq_alpha_x32", 7680, 4320, HapB200Codec_HapM, 32, 12, "ramp"),
            ("16k_hapq_x64", 16384, 16384, HapB200Codec_HapY, 64, 3, "opaque")]
    out = []
    stream = torch.cuda.Stream(device=dev)
    for name, w, h, codec, chunks, F, alpha in cfgs:
        try:
            rt = Roundtrip(lib, dev, w, h, codec, chunks, F, alpha=alpha)
            sp = stream.cuda_stream
            iters = 4 if w < 8000 else 2
            enc_ms = time_on_stream(torch, stream, lambda: rt.encode(sp), iters)
            dec_ms = time_on_stream(torch, stream, lambda: rt.decode(sp), iters)
            rt.check()
            # where one decode call of this batch spends its time (the library's own CUDA-event stage timer; not a bench value)
            torch.cuda.synchronize(dev)
            lib.set_stage_timing(True)
            lib.stage_times()
            with torch.cuda.stream(stream):
                rt.decode(sp)
            st = lib.stage_times()
            lib.set_stage_timing(False)
            dec_stages = {k: round(v[0], 4) for k, v in st.items() if v[1] and k in ("parse", "windows", "snappy_index", "snappy_decode", "collect")}
            frame_bytes = rt.mean_frame_bytes()
            tex_total = sum(rt.tex_bytes[: rt.ntex])
            enc_gbs = F * rt.rgba_bytes / enc_ms / 1e6
            dec_traffic = F * (frame_bytes + tex_total)
            out.append({"config": name, "frames_per_batch": F, "chunks": chunks, "ratio": frame_bytes / tex_total,
                        "encode": {"ms_per_frame": enc_ms / F, "fps": F / enc_ms * 1e3, "rgba_GBps": enc_gbs,
                                   "roofline_frac_rgba_read": enc_gbs / peak},
                        "decode": {"ms_per_frame": dec_ms / F, "fps": F / dec_ms * 1e3, "rgba_equiv_GBps": F * rt.rgba_bytes / dec_ms / 1e6,
                                   "traffic_GBps": dec_traffic / dec_ms / 1e6, "roofline_frac_frame_plus_texture": dec_traffic / dec_ms / 1e6 / peak,
                                   "stage_ms_per_batch": dec_stages}})
            del rt
            torch.cuda.empty_cache()
        except Exception as e:   # a configuration that does not fit must not hide the others
            out.append({"config": name, "error": repr(e)[:200]})
    return out


DUMP_SAMPLE = 1 << 22     # bytes sampled from the encoded frames and from the decoded textures: 16 MB of float32 each


def dump_outputs(out_dir, frames, used, cap, tex, tex_bytes):
    """--dump-outputs: what the last timed step handed back -- every frame's encoded length (frame_lengths.npy, float64), and
    a fixed, seeded sample of the encoded frame bytes (frame_bytes_sample.npy; -1 where a sampled position lies past its
    frame's end) and of the decoded texture bytes (texture_bytes_sample.npy), float32.  The inputs are seeded too, so two
    builds run with the same arguments can be compared file for file."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    n = used.numel()
    rng = np.random.default_rng(0)
    dev = frames.device
    pos = torch.from_numpy(np.sort(rng.integers(0, n * cap, DUMP_SAMPLE))).to(dev)
    fb = frames.view(-1)[pos].float()
    fb[(pos % cap) >= used[pos // cap]] = -1.0
    pos = torch.from_numpy(np.sort(rng.integers(0, n * tex_bytes, DUMP_SAMPLE))).to(dev)
    stride = (tex_bytes + 15) // 16 * 16
    tb = tex.view(-1)[(pos // tex_bytes) * stride + pos % tex_bytes].float()
    np.save(os.path.join(out_dir, "frame_lengths.npy"), used.double().cpu().numpy())
    np.save(os.path.join(out_dir, "frame_bytes_sample.npy"), fb.cpu().numpy())
    np.save(os.path.join(out_dir, "texture_bytes_sample.npy"), tb.cpu().numpy())


def run_gpu_arm(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist

    import hap_b200
    from hap_b200.lib import HapB200Codec_HapY

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = hap_b200.load()
    F = args.frames
    codec = HapB200Codec_HapY
    peak, peak_src = measured_peak_hbm()
    # the encoder appends its fragment index to every frame (hap_b200/csrc/hap_index.h: ~1 % of the frame; the reference
    # and FFmpeg ignore it) and the decoder uses it; --no-index times the frames laid out exactly as the reference writes them
    lib.set_option(lib.OPTION_WRITE_INDEX, 0 if args.no_index else 1)
    lib.set_option(lib.OPTION_USE_INDEX, 0 if args.no_index else 1)

    # ---- synthetic, device-resident input: F distinct frames per rank -------------------------------
    A = Roundtrip(lib, dev, W, H, codec, CHUNKS, F, first_index=rank * F)
    # two frame buffers: while the frames encoded in step i are being decoded (stream B), step i+1 already
    # encodes into the other buffer (stream A).  Every step encodes one batch and decodes one batch; the
    # decoded batch is the one the previous step encoded, i.e. a two-stage software pipeline over the stream.
    frames_buf = [A.frames, torch.empty_like(A.frames)]
    used = [A.used, torch.zeros_like(A.used)]
    stream = torch.cuda.Stream(device=dev)     # A: encode (and everything, when --no-overlap)
    stream_b = torch.cuda.Stream(device=dev)   # B: decode
    sp, spb = stream.cuda_stream, stream_b.cuda_stream
    overlap = not args.no_overlap
    encoded = [torch.cuda.Event() for _ in range(2)]   # buffer k holds a freshly encoded batch
    drained = [torch.cuda.Event() for _ in range(2)]   # buffer k has been decoded and may be overwritten
    state = {"n": 0}

    def encode_into(k, st):
        r = lib.encode_rgba_batch(A.rgba.data_ptr(), F, RGBA_BYTES, W, H, codec, 1, CHUNKS, frames_buf[k].data_ptr(), A.cap,
                                  used[k].data_ptr(), stream=st)
        assert r == 0, r

    def decode_from(k, st):
        A.decode(st, frames_buf[k].data_ptr(), used[k].data_ptr())

    def step():
        n = state["n"]
        k = n & 1
        if not overlap:
            encode_into(k, sp)
            decode_from(k, sp)
        else:
            if n >= 2:
                stream.wait_event(drained[k])          # the decode that read buffer k two steps ago is done
            encode_into(k, sp)
            encoded[k].record(stream)
            if n >= 1:
                stream_b.wait_event(encoded[k ^ 1])    # decode what the previous step encoded
                decode_from(k ^ 1, spb)
                drained[k ^ 1].record(stream_b)
        state["n"] = n + 1

    def drain():
        # decode the batch the last step encoded (overlap mode leaves one in flight)
        if overlap and state["n"] >= 1:
            k = (state["n"] - 1) & 1
            stream_b.wait_event(encoded[k])
            decode_from(k, spb)
        stream.wait_stream(stream_b)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    with torch.cuda.stream(stream):
        for _ in range(max(args.warmup, 3)):
            step()
        drain()
        barrier()
        A.check()
        state["n"] = 0
        launches0 = lib.launches()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        wall0 = time.time()
        e0.record(stream)
        # K steps = K batches encoded AND K batches decoded: in overlap mode the first timed step has nothing of
        # its own to decode yet, so the batch of the last step is decoded inside the timed region by drain()
        for _ in range(args.steps):
            step()
        drain()
        e1.record(stream)
        barrier()
        wall1 = time.time()
        launches = lib.launches() - launches0
        clocks = sampler.stop(wall0, wall1) if rank == 0 else None
        A.check()
        if args.dump_outputs and rank == 0:
            last = (state["n"] - 1) & 1
            dump_outputs(args.dump_outputs, frames_buf[last], used[last], A.cap, A.tex[0], A.tex_bytes[0])
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    ms_per_step = ms_total / args.steps
    value = world * F * RGBA_BYTES / (ms_per_step * 1e-3) / 1e9
    mean_frame = float(used[0].double().mean().item())

    # ---- end-to-end legs (every rank at once: the whole-job number at N GPUs): host-pointer C-ABI calls, one frame per
    #      call, pinned host buffers, PCIe copies inside the timed region.  `--e2e-threads` host threads per GPU keep that
    #      many frames in flight, the way a player or transcoder with a worker pool drives the codec (the reference is
    #      re-entrant; so is this library). ----------------------------------------------------------------------------
    e2e = e2e_rgba = None
    if not args.profile:
        import ctypes as C
        from concurrent.futures import ThreadPoolExecutor
        from hap_b200.abi import DECODE_CB, HapTextureFormat_YCoCg_DXT5

        FE, T = args.e2e_frames, max(1, args.e2e_threads)
        n_host = min(FE, F, 16)                      # distinct source frames in pinned host memory, cycled
        # host side of a deployment: the threads that feed a GPU and their pinned buffers sit on the GPU's own NUMA node
        # (PCIe DMA to the other socket's memory crosses the inter-socket link).  Linux exposes the node's CPUs per PCI device.
        numa_cpus, all_cpus = None, None
        if not args.no_numa:
            try:
                pr = torch.cuda.get_device_properties(local_rank)
                path = f"/sys/bus/pci/devices/{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0/local_cpulist"
                cpus = set()
                for part in open(path).read().strip().split(","):
                    lo, _, hi = part.partition("-")
                    cpus.update(range(int(lo), int(hi or lo) + 1))
                all_cpus = os.sched_getaffinity(0)
                cpus &= all_cpus
                if cpus and len(cpus) < len(all_cpus):
                    numa_cpus = cpus
                    os.sched_setaffinity(0, numa_cpus)      # this thread allocates (first-touches) the pinned buffers below
            except Exception:
                numa_cpus = None
        host_rgba = torch.empty((n_host, H, W, 4), dtype=torch.uint8).pin_memory()
        host_rgba.copy_(A.rgba[:n_host])
        # DXT textures of those frames (made by the block encoder once, outside the timed region): what a host
        # application hands to HapEncode
        dtex = torch.empty(n_host * DXT_BYTES, dtype=torch.uint8, device=dev)
        assert lib.block_encode_batch(A.rgba.data_ptr(), n_host, RGBA_BYTES, W, H, codec, dtex.data_ptr(), DXT_BYTES) == 0
        host_dxt = torch.empty((n_host, DXT_BYTES), dtype=torch.uint8).pin_memory()
        host_dxt.copy_(dtex.view(n_host, DXT_BYTES))
        del dtex
        host_frame = [torch.empty(A.cap, dtype=torch.uint8).pin_memory() for _ in range(T)]
        host_tex = [torch.empty(DXT_BYTES, dtype=torch.uint8).pin_memory() for _ in range(T)]

        def _cb(function, p, count, info):
            for i in range(count):
                function(p, i)
        cb = DECODE_CB(_cb)

        if numa_cpus:
            os.sched_setaffinity(0, all_cpus)               # (the buffers are placed; the main thread is free again)

        def worker_factory(use_rgba):
            def worker(w):
                if numa_cpus:
                    os.sched_setaffinity(0, numa_cpus)      # per thread on Linux
                usedc, fmtc = C.c_ulong(0), C.c_uint(0)
                h2d = d2h = 0
                for i in range(w, FE, T):
                    if use_rgba:
                        r = lib.lib.HapB200EncodeRGBA(host_rgba[i % n_host].data_ptr(), W, H, 4 * W, codec, 1, CHUNKS,
                                                      host_frame[w].data_ptr(), A.cap, C.byref(usedc))
                        h2d += RGBA_BYTES
                    else:
                        ins = (C.c_void_p * 1)(host_dxt[i % n_host].data_ptr())
                        r = lib._enc(1, ins, (C.c_ulong * 1)(DXT_BYTES), (C.c_uint * 1)(HapTextureFormat_YCoCg_DXT5), (C.c_uint * 1)(1),
                                     (C.c_uint * 1)(CHUNKS), host_frame[w].data_ptr(), A.cap, C.byref(usedc))
                        h2d += DXT_BYTES
                    assert r == 0, r
                    n = usedc.value
                    r = lib._dec(host_frame[w].data_ptr(), n, 0, cb, None, host_tex[w].data_ptr(), DXT_BYTES, C.byref(usedc), C.byref(fmtc))
                    assert r == 0 and usedc.value == DXT_BYTES, (r, usedc.value)
                    h2d += n
                    d2h += n + DXT_BYTES
                return h2d, d2h
            return worker

        pool = ThreadPoolExecutor(T)

        def e2e_leg(use_rgba, api):
            worker = worker_factory(use_rgba)

            def one():
                parts = list(pool.map(worker, range(T)))
                return sum(p[0] for p in parts), sum(p[1] for p in parts)
            for _ in range(2):
                one()
            barrier()
            t0 = time.perf_counter()
            iters = 3
            for _ in range(iters):
                h2d, d2h = one()
            torch.cuda.synchronize(dev)
            t = torch.tensor([(time.perf_counter() - t0) / iters], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)     # the slowest rank closes the step
            t = float(t.item())
            return {"value": world * FE * RGBA_BYTES / t / 1e9, "unit": "GB/s", "h2d_bytes_per_step": world * h2d,
                    "d2h_bytes_per_step": world * d2h, "frames_per_step": world * FE, "fps": world * FE / t, "host_threads": T * world,
                    "numa": (f"threads and pinned buffers on the GPU's NUMA node ({len(numa_cpus)} of {len(all_cpus)} CPUs)" if numa_cpus else "not bound"),
                    "api": api + f", pinned host buffers, one frame per call, {T} host threads per GPU, all {world} GPU(s) at once"}

        e2e = e2e_leg(False, "HapEncode(host DXT texture) + HapDecode(host frame -> host DXT): the reference's own API boundary")
        e2e_rgba = e2e_leg(True, "HapB200EncodeRGBA(host RGBA) + HapDecode(host frame -> host DXT)")
        del host_rgba, host_frame, host_tex, host_dxt
        pool.shutdown()

    # ---- N > 1 only, outside the timed region: the one step of a multi-GPU deployment that does cross GPUs -- delivering the
    #      encoded frames to the rank where the consumer sits (sharding.gatherv_frames_to_root: all-gather of the lengths +
    #      grouped ncclSend/ncclRecv of exactly the encoded bytes, NVLink).  64 frames of the batch per rank. ------------------
    delivery = None
    if world > 1 and not args.profile:
        from hap_b200 import sharding
        FD = min(F, 64)
        fview = frames_buf[0].view(F, A.cap)[:FD]
        uview = used[0][:FD]
        ring = torch.empty((world, FD, A.cap), dtype=torch.uint8, device=dev) if rank == 0 else None
        with torch.cuda.stream(stream):
            for _ in range(2):
                _, lengths = sharding.gatherv_frames_to_root(fview, uview, 0, ring)
            barrier()
            d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            d0.record(stream)
            for _ in range(3):
                _, lengths = sharding.gatherv_frames_to_root(fview, uview, 0, ring)
            d1.record(stream)
            barrier()
            dms = torch.tensor([d0.elapsed_time(d1) / 3], dtype=torch.float64, device=dev)
            dist.all_reduce(dms, op=dist.ReduceOp.MAX)
        moved = int(lengths.sum() - lengths[0].sum())
        if rank == 0:
            ok = all(torch.equal(ring[r, i, : int(lengths[r, i])][:64], ring[r, i, :64]) for r in range(world) for i in (0, FD - 1))
            delivery = {"what": f"{FD} encoded frames per rank delivered to rank 0",
                        "nccl_gatherv": {"what": "frames already encoded in local memory: all-gather of lengths + grouped ncclSend/ncclRecv, device to device",
                                         "ms": float(dms.item()), "nvlink_bytes": moved, "nvlink_GBps_into_rank0": moved / (float(dms.item()) * 1e-3) / 1e9,
                                         "frames_per_s": world * FD / (float(dms.item()) * 1e-3), "ok": bool(ok)}}
        del ring
        # the library's own way (include/hap_b200.h, HapB200Ring*): every rank ENCODES its frames straight into a delivery ring
        # in rank 0's memory (CUDA IPC peer mapping): the frame-layout kernel's stores go over NVLink, nothing passes over the
        # encoded bytes a second time.  Timed: encode of FD frames into the ring + publish on every rank, rank 0 waiting for
        # every slot; next to it the same encode into local memory.
        HEADER = 4096
        slot_bytes = HEADER + FD * A.cap
        handle = torch.zeros(lib.RING_HANDLE_BYTES, dtype=torch.uint8, device=dev)
        ring_ptr, ring_up = 0, 1
        if rank == 0:
            rr, ring_ptr, hb = lib.ring_create(local_rank, world * slot_bytes)
            ring_up = int(rr == 0)
            if ring_up:
                handle.copy_(torch.frombuffer(bytearray(hb), dtype=torch.uint8))
        dist.broadcast(handle, 0)
        if rank != 0:
            rr, ring_ptr = lib.ring_open(local_rank, handle.cpu().numpy().tobytes())
            ring_up = int(rr == 0 and ring_ptr != 0)
        agreed = torch.tensor([ring_up], dtype=torch.int32, device=dev)
        dist.all_reduce(agreed, op=dist.ReduceOp.MIN)       # every rank takes the same branch below
        ring_up = int(agreed.item())
        my_slot = ring_ptr + rank * slot_bytes
        consumer = torch.cuda.Stream(device=dev)
        seq = {"n": 0}

        def into_ring():
            seq["n"] += 1
            assert lib.encode_rgba_batch(A.rgba.data_ptr(), FD, RGBA_BYTES, W, H, codec, 1, CHUNKS, my_slot + HEADER, A.cap, my_slot + 64, stream=stream.cuda_stream) == 0
            assert lib.ring_publish(local_rank, my_slot, seq["n"], stream=stream.cuda_stream) == 0
            if rank == 0:
                for q in range(world):
                    assert lib.ring_wait(local_rank, ring_ptr + q * slot_bytes, seq["n"], 0, stream=consumer.cuda_stream) == 0

        def into_local():
            assert lib.encode_rgba_batch(A.rgba.data_ptr(), FD, RGBA_BYTES, W, H, codec, 1, CHUNKS, frames_buf[0].data_ptr(), A.cap, used[0].data_ptr(), stream=stream.cuda_stream) == 0

        def timed_ms(fn, reps=3):
            with torch.cuda.stream(stream):
                fn()
                barrier()
                a0, a1, c1 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                a0.record(stream)
                for _ in range(reps):
                    fn()
                a1.record(stream)
                c1.record(consumer)
                barrier()
                t = torch.tensor([max(a0.elapsed_time(a1), a0.elapsed_time(c1)) / reps], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        if not ring_up:
            if rank == 0:
                delivery["ring"] = {"error": "the delivery ring could not be set up on every rank (HapB200RingCreate / HapB200RingOpen: CUDA IPC between these processes)"}
                if ring_ptr:
                    lib.ring_destroy(local_rank, ring_ptr)
            elif ring_ptr:
                lib.ring_close(local_rank, ring_ptr)
        ms_ring, ms_local = (timed_ms(into_ring), timed_ms(into_local)) if ring_up else (None, None)
        if rank == 0 and ring_up:
            class _Ext:
                def __init__(self, ptr, nb):
                    self.__cuda_array_interface__ = {"shape": (nb,), "typestr": "|u1", "data": (ptr, False), "version": 2}
            rt = torch.as_tensor(_Ext(ring_ptr, world * slot_bytes), device=dev)
            rl = torch.stack([rt[q * slot_bytes + 64: q * slot_bytes + 64 + 8 * FD].view(torch.int64).cpu() for q in range(world)])
            ring_ok = bool(torch.equal(rl, lengths))     # every rank's frames arrived with the lengths the NCCL leg moved
            delivery["ring"] = {"what": "frames ENCODED straight into a delivery ring in rank 0's memory (HapB200Ring*: CUDA IPC peer mapping, the frame-layout "
                                        "kernel stores over NVLink, release-store flags, rank 0 waits by stream memory operations); no collective",
                                "encode_into_ring_ms": ms_ring, "encode_into_local_memory_ms": ms_local, "delivery_overhead_ms": ms_ring - ms_local,
                                "nvlink_bytes": moved, "nvlink_GBps_into_rank0": moved / (ms_ring * 1e-3) / 1e9,
                                "frames_per_s": world * FD / (ms_ring * 1e-3), "lengths_equal_nccl_leg": ring_ok}
            del rt
        barrier()
        if ring_up and rank != 0:
            assert lib.ring_close(local_rank, ring_ptr) == 0
        barrier()
        if ring_up and rank == 0:
            assert lib.ring_destroy(local_rank, ring_ptr) == 0

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- roofline leg: per-stage CUDA events (not part of the timed region) ------------------------------
    lib.set_stage_timing(True)
    lib.stage_times()
    overlap_was, overlap = overlap, False   # stage timing needs the kernels one after another
    with torch.cuda.stream(stream):
        for _ in range(3):
            step()
    overlap = overlap_was
    st = lib.stage_times()
    lib.set_stage_timing(False)
    per_step = {k: v[0] / 3 for k, v in st.items()}
    # one batch = one launch of every stage's main kernel (the decode stages launch a second, normally empty, repair pass:
    # its few microseconds are counted with the stage)
    stage_ms = dict(per_step)
    dominant = max(stage_ms, key=lambda k: per_step[k])
    alg_bytes = lib.stage_algorithmic_bytes(F, RGBA_BYTES, DXT_BYTES, mean_frame)
    dom_ms = stage_ms[dominant]
    achieved = alg_bytes[dominant] / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        try:
            per_frame = json.load(open(tpath)).get("per_frame_bytes", {}).get(dominant)
            traffic = per_frame * F if per_frame is not None else None   # measured per frame (ncu), scaled to this launch
        except Exception:
            traffic = None
    stage_frac = {k: (alg_bytes[k] / (stage_ms[k] * 1e-3) / 1e9 / peak if stage_ms[k] > 0 else None) for k in stage_ms}
    if not args.no_index:
        stage_frac["snappy_index"] = None       # frames carry their index: the kernel is launched on an empty list
    roofline = {"bound": "hbm", "kernel": dominant, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes[dominant], "ms_per_launch": dom_ms,
                "stage_ms_per_step": per_step, "stage_frac_of_hbm": stage_frac}
    if args.profile:
        emit({"profile_only": True, "ms_per_step": ms_per_step, "value": value, "roofline": roofline})
        return

    # encode-only / decode-only of the headline batch (one stream, CUDA events): the two north-star targets separately
    enc_ms = time_on_stream(torch, stream, lambda: encode_into(0, sp), 3)
    dec_ms = time_on_stream(torch, stream, lambda: decode_from(0, sp), 3)
    split = {"encode": {"ms_per_batch": enc_ms, "fps": F / enc_ms * 1e3, "rgba_GBps": F * RGBA_BYTES / enc_ms / 1e6,
                        "roofline_frac_rgba_read": F * RGBA_BYTES / enc_ms / 1e6 / peak, "target": 0.70},
             "decode": {"ms_per_batch": dec_ms, "fps": F / dec_ms * 1e3, "rgba_equiv_GBps": F * RGBA_BYTES / dec_ms / 1e6,
                        "traffic_GBps": F * (mean_frame + DXT_BYTES) / dec_ms / 1e6,
                        "roofline_frac_frame_plus_texture": F * (mean_frame + DXT_BYTES) / dec_ms / 1e6 / peak, "target": 0.80}}

    extra = {}
    if delivery is not None:
        extra["delivery_to_rank0"] = delivery
    if not args.no_index:
        lib.set_option(lib.OPTION_USE_INDEX, 0)
        ms_noix = time_on_stream(torch, stream, lambda: decode_from(0, sp), 3)
        lib.set_option(lib.OPTION_USE_INDEX, 1)
        extra["own_stream_decode_without_index"] = {
            "what": "the same batch decoded with the embedded index ignored (snappy_index_kernel derives it from the streams)",
            "ms_per_batch": ms_noix, "fps": F / ms_noix * 1e3, "traffic_GBps": F * (mean_frame + DXT_BYTES) / ms_noix / 1e6,
            "roofline_frac_frame_plus_texture": F * (mean_frame + DXT_BYTES) / ms_noix / 1e6 / peak}
    if world == 1 and not args.no_extra:
        del frames_buf, used
        extra["configs"] = extra_config_lines(lib, torch, dev, peak)

    # ---- CPU baseline leg (bounded) + decode of the frames the REFERENCE encoder made there -----------------
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            r = reference_cpu_path(3, 1, keep_frames=64)
            cpu = {"value": r["value"], "unit": "GB/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"],
                   "detail": {k: v for k, v in r.items() if k not in ("value", "sample", "_frames", "cores", "kind")}}
            buf, cap_r, used_r, texs = r["_frames"]
            n0 = len(used_r)
            rep = max(1, 256 // n0)          # the distinct frames, repeated on the device to a batch that fills the GPU
            n = n0 * rep
            d_frames = torch.from_numpy(buf).to(dev).repeat(rep)
            d_used = torch.tensor(list(used_r) * rep, dtype=torch.int64, device=dev)
            B = Roundtrip.__new__(Roundtrip)
            B.lib, B.F, B.cap, B.chunks, B.ntex, B.tex_bytes = lib, n, cap_r, CHUNKS, 1, [DXT_BYTES, 0]
            B.tex = [torch.empty(n * DXT_BYTES, dtype=torch.uint8, device=dev)]
            B.tex_used = torch.zeros(n, dtype=torch.int64, device=dev)
            B.fmts = torch.zeros(n, dtype=torch.int32, device=dev)
            B.res = torch.zeros(n, dtype=torch.int32, device=dev)
            B.used = d_used
            ms_ref = time_on_stream(torch, stream, lambda: B.decode(sp, d_frames.data_ptr(), d_used.data_ptr()), 5)
            B.check()
            import numpy as np
            got = B.tex[0].view(n, DXT_BYTES).cpu().numpy()
            assert all((got[i] == texs[i % n0]).all() for i in range(n)), "GPU decode of reference-made frames differs from the payload"
            lib.set_stage_timing(True)
            lib.stage_times()
            with torch.cuda.stream(stream):
                for _ in range(3):
                    B.decode(sp, d_frames.data_ptr(), d_used.data_ptr())
            st_ref = lib.stage_times()
            lib.set_stage_timing(False)
            fb = float(sum(used_r)) / n0
            extra["ref_stream_decode"] = {
                "what": f"HapB200DecodeBatch on {n} 4K Hap Q frames ({CHUNKS} chunks; {n0} distinct, made by the {r['kind']} encoder: "
                        "byte-granular Google-Snappy streams), device-resident, bytes compared with the payload",
                "ms_per_frame": ms_ref / n, "fps": n / ms_ref * 1e3, "rgba_equiv_GBps": n * RGBA_BYTES / ms_ref / 1e6,
                "traffic_GBps": n * (fb + DXT_BYTES) / ms_ref / 1e6, "roofline_frac_frame_plus_texture": n * (fb + DXT_BYTES) / ms_ref / 1e6 / peak,
                "ratio": fb / DXT_BYTES,
                "stage_ms_per_batch": {k: v[0] / 3 for k, v in st_ref.items() if v[0] > 0}}
        except Exception as e:  # the oracle is a checker; its absence must not hide the GPU number
            cpu = {"value": None, "unit": "GB/s", "cores": os.cpu_count(), "kind": "port", "sample": f"unavailable: {e!r}"[:300]}

    line = {
        "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic", "config": CONFIG,
        "run": {"frames_per_gpu_per_step": F, "rgba_GB_per_step_per_gpu": F * RGBA_BYTES / 1e9, "compression_ratio": mean_frame / DXT_BYTES,
                "parallelism": f"frames sharded over {world} gpu(s), no collective on the data path",
                "pipelining": "decode(batch i) on stream B overlaps encode(batch i+1) on stream A" if overlap else "none",
                "fragment_index": "off (frames byte-identical in layout to the reference's)" if args.no_index else
                                  "on (trailing private section, ~1 % of the frame, ignored by the reference and FFmpeg)"},
        "fps": world * F / (ms_per_step * 1e-3),
        "encode_decode_split": split,
        "clocks": clocks, "e2e": e2e, "e2e_rgba": e2e_rgba, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu,
        "extra": extra,
    }
    emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line: dict):
    """The ONE JSON line, on the process's real stdout (see main(): fd 1 itself is pointed at stderr while the
    run lasts, because NCCL prints its version banner straight to fd 1 when the first communicator is made)."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="4k_hapq", choices=["4k_hapq", "16k_stream"])
    ap.add_argument("--frames", type=int, default=444, help="device-resident frames per GPU per step")
    ap.add_argument("--e2e-frames", type=int, default=64)
    ap.add_argument("--e2e-threads", type=int, default=16)
    ap.add_argument("--no-numa", action="store_true", help="e2e legs: do not bind host threads / pinned buffers to the GPU's NUMA node")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the per-configuration encode-only / decode-only lines")
    ap.add_argument("--profile", action="store_true", help="short run for ncu: skip the e2e, extra and CPU legs")
    ap.add_argument("--no-overlap", action="store_true", help="encode and decode of a batch back to back on one stream")
    ap.add_argument("--no-index", action="store_true", help="frames without the trailing fragment index section (decoder indexes on the fly)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last step computed (encoded frame "
                                                          "lengths, sampled frame and texture bytes) as .npy files into DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "4k_hapq"):
        ap.error("--dump-outputs applies to the 4k_hapq workload of the b200 implementation")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    if args.workload == "16k_stream":
        from hap_b200 import stream_bench
        stream_bench.run(args, rank, local_rank, world, emit, ClockSampler, measured_peak_hbm)
        return
    run_gpu_arm(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
