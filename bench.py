#!/usr/bin/env python3
"""bench.py -- SELA hot path on B200: encode + decode MSamples/s (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

A step = one pass of the hot path over one batch: fused encode of the batch (PCM ->
descriptors + Rice words) followed by decode of what was just produced (-> PCM).
Workload at every N: BASELINE.json configs[1]/[2] per GPU -- 44.1 kHz 16-bit stereo,
10 min of synthetic sine+noise (12 919 frames, 52.9 M samples) -- i.e. weak scaling,
each rank codes its own file (seed 1+rank), no data-path collective (frames are
independent; SURVEY.md 8e).

  value   device-resident: PCM already in HBM, CUDA-event timed, max over ranks.
  e2e     same metric through the host-buffer C ABI (selab200_encode_frames /
          selab200_decode_frames) from pinned host memory, H2D + D2H inside the timing.
  --impl reference   the reference's own multithreaded CPU path (oracle/_ref when it was
          compiled from /root/reference, else the plain-C port in oracle/) on the host cores.
"""
import argparse
import ctypes as C
import json
import os
import pathlib
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

FRAME = 2048
SAMPLE_RATE, CHANNELS, SECONDS = 44100, 2, 600
WORKLOAD = "44.1kHz 16-bit stereo 10min synthetic sine+noise (BASELINE configs[1]+[2]), encode then decode"
METRIC = "encode+decode MSamples/s"


def measured_peak_hbm():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi sampled every 50 ms from before the warm-up; only samples whose timestamp falls
    inside the timed region [t0, t1] are kept."""
    FIELDS = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.FIELDS,
                                       "--format=csv,noheader,nounits", "-lms", "50"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self, t0, t1):
        import datetime
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.split(", ") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        total = 0
        for r in rows:
            try:
                ts = datetime.datetime.strptime(r[0].strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()
                vals = (float(r[1]), float(r[2]), float(r[3]))
            except (ValueError, IndexError):
                continue
            total += 1
            if not (t0 - 0.05 <= ts <= t1 + 0.05):
                continue
            sm.append(vals[0]); smax.append(vals[1]); power.append(vals[2])
            for n, v in zip(names, r[4:8]):
                if v.strip().lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "samples_total": total,
                "reasons": sorted(reasons)}


def workload_config(n_frames, n_samples):
    """The `config` object of BOTH arms (the driver compares them): what one GPU's workload is."""
    return {"workload": WORKLOAD, "frames_per_gpu": n_frames, "samples_per_gpu": n_samples,
            "l2": "no flush: per step the kernels stream the PCM, the word arena and the residue workspace of the "
                  "whole file (about 390 MB), larger than the 126 MB L2"}


def source_hash():
    """Hash of the kernel sources: ties the ncu-derived numbers in profiles/traffic.json to the code that ran."""
    import hashlib
    h = hashlib.sha256()
    for f in sorted((ROOT / "sela_b200" / "csrc").glob("*")):
        h.update(f.name.encode())
        h.update(f.read_bytes())
    return h.hexdigest()[:16]


def measured_profile(kernel):
    """What the committed ncu capture says about `kernel` (profiles/traffic.json): DRAM bytes per launch, pipe
    utilisation.  Returns (entry or None, stale flag): stale = the kernel sources changed since the capture."""
    p = ROOT / "profiles" / "traffic.json"
    try:
        doc = json.loads(p.read_text())
        e = doc[kernel]
        return e, doc.get("source_hash") != source_hash()
    except Exception:
        return None, True


def measured_traffic(kernel):
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture (cannot be taken
    inside the bench: a number measured under a profiler is never a bench value)."""
    p = ROOT / "profiles" / "traffic.json"
    try:
        return int(json.loads(p.read_text())[kernel]["traffic"])
    except Exception:
        return None



def rice_decode_roofline(codec, n_frames, n_words, dev, peak, tiles=(1, 16)):
    """The Rice-decode kernel (K5) on its own, timed here with CUDA events through
    selab200_rice_decode_frames_device: BASELINE's batch, and the same streams tiled to a batch that fills the
    machine.  Algorithmic bytes (SURVEY.md 8d): residue words read + 4 B per decoded sample written."""
    import torch
    from sela_b200 import _lib
    L = _lib.lib()
    descs = codec.descs.cpu().numpy().view(_lib.DESC_DTYPE).copy()
    res_words = int(descs["res_words"].astype(np.int64).sum())
    words = codec.words[:n_words]
    out = {}
    for tile in tiles:
        d = np.tile(descs, tile)
        for r in range(1, tile):
            sl = slice(r * descs.size, (r + 1) * descs.size)
            d["refl_offset"][sl] += r * n_words
            d["res_offset"][sl] += r * n_words
        d_descs = torch.from_numpy(d.view(np.uint8).reshape(-1)).to(dev)
        d_words = torch.cat([words.repeat(tile), torch.zeros(8, dtype=words.dtype, device=dev)])
        n_sub = d.size
        res = torch.empty(n_sub * FRAME, dtype=torch.int32, device=dev)
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        stream = torch.cuda.current_stream(dev).cuda_stream

        def run():
            _lib.check(L.selab200_rice_decode_frames_device(d_descs.data_ptr(), n_frames * tile, CHANNELS, d_words.data_ptr(),
                                                            n_words * tile, res.data_ptr(), status.data_ptr(), C.c_void_p(stream)))
        for _ in range(3):
            run()
        torch.cuda.synchronize(dev)
        reps = 10 if tile == 1 else 4
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev[0].record()
        for _ in range(reps):
            run()
        ev[1].record()
        torch.cuda.synchronize(dev)
        ms = ev[0].elapsed_time(ev[1]) / reps
        flagged = C.c_uint32(0)
        _lib.check(L.selab200_rice_decode_flagged(C.addressof(flagged)))
        alg = res_words * tile * 4 + n_sub * FRAME * 4
        out["streams_%d" % n_sub] = {
            "streams": n_sub, "ms": ms, "gsamples_s": n_sub * FRAME / ms / 1e6, "achieved": alg / ms / 1e6, "unit": "GB/s",
            "peak": peak, "frac": alg / ms / 1e6 / peak, "algorithmic_bytes": alg, "status": int(status.item()),
            "streams_redone_by_general_parser": int(flagged.value)}
        del d_descs, d_words, res
    return out


def pcie_probe(dev, nbytes=128 << 20):
    """Pinned-memory copy rates of this box (they differ by 2x between boxes; the e2e number is PCIe bound)."""
    import torch
    h = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    d = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    res = {}
    for name, (dst, src) in (("h2d_gbs", (d, h)), ("d2h_gbs", (h, d))):
        dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(3):
            dst.copy_(src, non_blocking=True)
        b.record()
        torch.cuda.synchronize(dev)
        res[name] = 3 * nbytes / a.elapsed_time(b) / 1e6
    # both directions at once, as the pipelined calls drive the link (on some boxes each direction then runs slower)
    h2, d2 = torch.empty(nbytes, dtype=torch.uint8).pin_memory(), torch.empty(nbytes, dtype=torch.uint8, device=dev)
    s_up, s_down = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    torch.cuda.synchronize(dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    with torch.cuda.stream(s_up):
        ev[0].record()
        for _ in range(3):
            d.copy_(h, non_blocking=True)
        ev[1].record()
    with torch.cuda.stream(s_down):
        ev[2].record()
        for _ in range(3):
            h2.copy_(d2, non_blocking=True)
        ev[3].record()
    torch.cuda.synchronize(dev)
    res["h2d_gbs_both_directions"] = 3 * nbytes / ev[0].elapsed_time(ev[1]) / 1e6
    res["d2h_gbs_both_directions"] = 3 * nbytes / ev[2].elapsed_time(ev[3]) / 1e6
    return res


def sharded_block(args, rank, world, dev, dist):
    """BASELINE configs[3] and [4] on the N GPUs of this run.
      config4: ONE 48 kHz 8-channel file coded by all ranks: PCM scattered from rank 0 over NCCL, every rank
               encodes its contiguous block of frames, coded subframes gathered on rank 0 (offsets re-based);
               then the reverse for decode.  Checked against rank 0 coding the whole file alone.
      config5: a batch of independent 3-minute stereo files, 1024 / N per rank, coded file by file."""
    import torch
    from sela_b200 import distributed as sd, synth
    from sela_b200.device import DeviceCodec
    out = {}
    # ---------------- config 4 ----------------
    ch, rate = 8, 48000
    base_min, reps = 3, 20 if not args.sharded_minutes else max(1, args.sharded_minutes // 3)
    n_base = (rate * 60 * base_min) // FRAME
    n_frames = n_base * reps
    per = FRAME * ch
    if rank == 0:
        base = torch.from_numpy(synth.sine_noise(rate, ch, n_frames=n_base, seed=2).reshape(-1))
        pcm_dev = torch.empty(n_frames * per, dtype=torch.int16, device=dev)
        base_pinned = base.pin_memory()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        base_dev = base_pinned.to(dev, non_blocking=True)
        torch.cuda.synchronize(dev)
        h2d_s = time.perf_counter() - t0
        del base_pinned
        for r in range(reps):
            pcm_dev[r * n_base * per:(r + 1) * n_base * per].copy_(base_dev)
        del base_dev
    else:
        pcm_dev, h2d_s = None, 0.0
    if dist:
        dist.barrier()
    if dist:
        # first pass of each: NCCL sets its peer connections up and the allocator grows; of the two warm passes
        # that follow, the one with the smaller total is reported (a single pass now and then stalls for tens of ms)
        total = lambda tt: sum(v for k, v in tt.items() if k.endswith("_ms"))
        sd.encode_sharded_device(pcm_dev, n_frames, ch, root=0)
        (d_all2, w_all2), t_enc2 = sd.encode_sharded_device(pcm_dev, n_frames, ch, root=0)
        (d_all3, w_all3), t_enc3 = sd.encode_sharded_device(pcm_dev, n_frames, ch, root=0)
        if rank == 0:
            same_again = bool(torch.equal(d_all2, d_all3)) and bool(torch.equal(w_all2, w_all3))
        del d_all3, w_all3
        sd.decode_sharded_device(d_all2, w_all2, n_frames, ch, root=0)
        pcm_back, t_dec = sd.decode_sharded_device(d_all2, w_all2, n_frames, ch, root=0)
        _, t_dec3 = sd.decode_sharded_device(d_all2, w_all2, n_frames, ch, root=0)
        passes = torch.tensor([total(t_enc2), total(t_enc3), total(t_dec), total(t_dec3)], dtype=torch.float64, device=dev)
        dist.all_reduce(passes, op=dist.ReduceOp.MAX)          # every rank must pick the same pass
        pe = passes.tolist()
        if pe[1] < pe[0]:
            t_enc2 = t_enc3
        if pe[3] < pe[2]:
            t_dec = t_dec3
    else:
        t_enc2 = t_dec = None
    c4 = {"workload": "48 kHz 16-bit 8-channel, %d min (%d x the %d-minute seed-2 synthetic), one file across %d GPU(s)" % (
        base_min * reps, reps, base_min, world), "frames": n_frames, "samples": n_frames * per}
    if rank == 0:
        single = DeviceCodec(n_frames, ch, device=dev.index)
        single.encode(pcm_dev)
        torch.cuda.synchronize(dev)
        (_, ms1) = sd._timed(lambda: single.encode(pcm_dev), dev)
        single.check_status()
        nw1 = int(single.words_used.item())
        out1 = torch.empty_like(pcm_dev)
        single.decode(out1, nw1)
        torch.cuda.synchronize(dev)
        (_, ms1d) = sd._timed(lambda: single.decode(out1, nw1), dev)
        single.check_status()
        c4["single_gpu"] = {"encode_ms": ms1, "decode_ms": ms1d, "encode_msamples_s": n_frames * per / ms1 / 1e3,
                            "decode_msamples_s": n_frames * per / ms1d / 1e3, "words": nw1,
                            "decode_equals_source_samples": int((out1 == pcm_dev).sum().item()), "samples": n_frames * per}
        if dist:
            same = bool(torch.equal(d_all2, single.descs)) and w_all2.numel() == nw1 and bool(torch.equal(w_all2, single.words[:nw1]))
            c4["bytes_identical_to_single_gpu"] = same and same_again
            c4["decode_identical_to_single_gpu"] = bool(torch.equal(pcm_back, out1))
        c4["root_upload_gbs"] = base.numel() * 2 / h2d_s / 1e9
        del single, out1
    if dist:
        # max over ranks of every phase, wall time of the whole sharded call = sum of the phase maxima
        keys_e, keys_d = ("scatter_ms", "encode_ms", "gather_ms"), ("scatter_ms", "decode_ms", "gather_ms")
        t = torch.tensor([t_enc2[k] for k in keys_e] + [t_dec[k] for k in keys_d], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        v = t.tolist()
        c4["nccl_encode"] = dict(zip(keys_e, v[:3]))
        c4["nccl_decode"] = dict(zip(keys_d, v[3:]))
        c4["nccl_encode"]["msamples_s"] = n_frames * per / sum(v[:3]) / 1e3
        c4["nccl_encode"]["msamples_s_kernels_only"] = n_frames * per / v[1] / 1e3
        c4["nccl_decode"]["msamples_s"] = n_frames * per / sum(v[3:]) / 1e3
        c4["nccl_decode"]["msamples_s_kernels_only"] = n_frames * per / v[4] / 1e3
        c4["note"] = ("scatter/gather move PCM (2 B/sample) and coded words between HBMs over NVLink; rank 0's own "
                      "PCIe upload/download is not in these times")
    out["config4"] = c4
    del pcm_dev
    torch.cuda.empty_cache()
    # ---------------- config 5 ----------------
    files_total, distinct = 1024, 8
    file_frames = (44100 * 180) // FRAME                       # 3 875 whole frames of a 3-minute file (the tail is dropped)
    fs = FRAME * 2 * file_frames
    bank = torch.empty(distinct * fs, dtype=torch.int16, device=dev)
    if rank == 0:
        for i in range(distinct):
            bank[i * fs:(i + 1) * fs].copy_(torch.from_numpy(synth.sine_noise(44100, 2, n_frames=file_frames, seed=i).reshape(-1)))
    if dist:
        dist.broadcast(bank.view(torch.uint8), 0)      # (NCCL has no int16)
    mine = files_total // world + (1 if rank < files_total % world else 0)
    codec = DeviceCodec(file_frames, 2, device=dev.index)
    outp = torch.empty(fs, dtype=torch.int16, device=dev)

    def code_file(i):
        pcm = bank[(i % distinct) * fs:(i % distinct + 1) * fs]
        codec.encode(pcm)
        return pcm
    nw = []
    for i in range(distinct):                                     # warm-up + the word counts the decoder needs
        code_file(i)
        torch.cuda.synchronize(dev)
        nw.append(int(codec.words_used.item()))
    ok = True
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    if dist:
        dist.barrier()
    torch.cuda.synchronize(dev)
    ev[0].record()
    for i in range(mine):
        code_file(i)
    ev[1].record()
    for i in range(mine):
        code_file(i)                                              # (the decoder reads what the encoder just wrote)
        codec.decode(outp, nw[i % distinct])
    ev[2].record()
    torch.cuda.synchronize(dev)
    codec.check_status()
    ok = bool(torch.equal(outp, bank[((mine - 1) % distinct) * fs:((mine - 1) % distinct + 1) * fs])) if mine else True
    enc_ms = ev[0].elapsed_time(ev[1])
    dec_ms = ev[1].elapsed_time(ev[2]) - enc_ms                   # second loop = encode + decode
    t = torch.tensor([enc_ms, dec_ms, 0.0 if ok else 1.0], dtype=torch.float64, device=dev)
    if dist:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    enc_ms, dec_ms, bad = t.tolist()
    total = files_total * fs
    out["config5"] = {
        "workload": "1024 independent 3-minute 44.1 kHz stereo files (%d distinct synthetic files, seeds 0..%d, reused), %s per rank, "
                    "one encode and one decode call per file, device resident" % (distinct, distinct - 1, "%d or %d" % (files_total // world, -(-files_total // world)) if files_total % world else str(files_total // world)),
        "files": files_total, "frames_per_file": file_frames, "samples": total,
        "encode_ms": enc_ms, "decode_ms": dec_ms, "encode_msamples_s": total / enc_ms / 1e3, "decode_msamples_s": total / dec_ms / 1e3,
        "encode_decode_msamples_s": total / (enc_ms + dec_ms) / 1e3, "round_trip_bit_exact": bad == 0.0}
    return out


_REAL_STDOUT = []


def emit_line(line):
    """Print the result line on the process's real stdout (see the fd juggling around NCCL init)."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT:
        sys.stdout.flush()
        os.write(_REAL_STDOUT[0], data)
    else:
        sys.stdout.write(data.decode())
        sys.stdout.flush()


def make_pcm(seed):
    from sela_b200 import synth
    return synth.sine_noise(SAMPLE_RATE, CHANNELS, seconds=SECONDS, seed=seed)


DUMP_FRAMES = 1024


def dump_outputs(path, descs, words, pcm_out):
    """--dump-outputs: what a caller of the timed path received from its last step, so that two builds can be
    compared output for output.  The workload's words and PCM run to hundreds of MB, so those two files hold a
    fixed sample of frames (seed 0; it depends only on the frame count), in frame order:
      descs.npy        float64 [subframes, 12]     every descriptor, fields in DESC_DTYPE order
      words.npy        float64 [n]                 each sampled frame's Rice words, subframe by subframe
      pcm_decoded.npy  float32 [frames*2048, ch]   the decoded PCM of the sampled frames"""
    n_frames = pcm_out.size // (FRAME * CHANNELS)
    frames = np.sort(np.random.default_rng(0).choice(n_frames, min(n_frames, DUMP_FRAMES), replace=False))
    sub = (frames[:, None] * CHANNELS + np.arange(CHANNELS)).reshape(-1)
    spans = [(int(descs[i][o]), int(descs[i][n])) for i in sub
             for o, n in (("refl_offset", "refl_words"), ("res_offset", "res_words"))]
    out = {
        "descs": np.stack([descs[f].astype(np.float64) for f in descs.dtype.names], axis=1),
        "words": np.concatenate([words[a:a + n] for a, n in spans]).astype(np.float64),
        "pcm_decoded": pcm_out.reshape(n_frames, FRAME, CHANNELS)[frames].reshape(-1, CHANNELS).astype(np.float32),
    }
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    os.makedirs(path, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), a)


def cpu_reference_leg(pcm, target_seconds=8.0):
    """Time the reference's multithreaded CPU coder on a bounded sample of the workload."""
    import oracle_lib as ol
    O = ol.best()
    n_frames = pcm.shape[0] // FRAME
    probe = min(n_frames, 256)
    t = O.time_encode(pcm[:probe * FRAME], CHANNELS)
    rate = probe / max(t, 1e-6)
    sample_frames = int(max(probe, min(n_frames, rate * target_seconds / 3)))
    sample = pcm[:sample_frames * FRAME]
    descs, words = O.encode_frames(sample, CHANNELS)
    te = statistics.median(O.time_encode(sample, CHANNELS) for _ in range(3))
    td = statistics.median(O.time_decode(descs, words, CHANNELS) for _ in range(3))
    n_samples = sample_frames * FRAME * CHANNELS
    info = {
        "value": n_samples / (te + td) / 1e6, "unit": "MSamples/s", "cores": O.cores, "kind": O.kind,
        "sample": "first %d of %d frames (%.1f s of audio), median of 3; timed: %s" % (
            sample_frames, n_frames, sample_frames * FRAME / SAMPLE_RATE,
            "sela::Encoder/Decoder::processFrames only" if O.kind == "reference" else "oracle port batch calls"),
        "encode_msamples_s": n_samples / te / 1e6, "decode_msamples_s": n_samples / td / 1e6,
        "seconds_per_pass": te + td,
    }
    return info, (sample_frames, descs, words)


def run_reference(args, rank, world):
    """The reference's own multithreaded CPU coder (sela::Encoder/Decoder::processFrames of oracle/_ref, or the
    plain-C port when the reference was not compiled) on the host cores.  A step = encode + decode of a
    BOUNDED SAMPLE of the workload (the first frames of the file; frames are independent, so the rate is the
    whole file's), sized by a probe so that warm-up + steps end within minutes on any box."""
    if rank != 0:
        return
    import oracle_lib as ol
    O = ol.best()
    pcm = make_pcm(1)
    n_frames = pcm.shape[0] // FRAME
    n_samples_file = n_frames * FRAME * CHANNELS
    probe = min(n_frames, 512)
    t_probe = O.time_encode(pcm[:probe * FRAME], CHANNELS)
    d_p, w_p = O.encode_frames(pcm[:probe * FRAME], CHANNELS)
    t_probe += O.time_decode(d_p, w_p, CHANNELS)
    rate = probe / max(t_probe, 1e-6)                     # frames per second, encode + decode
    budget = 90.0 / max(1, args.steps + args.warmup)      # seconds per step
    sample_frames = int(max(min(probe, n_frames), min(n_frames, rate * min(budget, 2.0))))
    sample = pcm[:sample_frames * FRAME]
    descs, words = O.encode_frames(sample, CHANNELS)
    n_samples = sample_frames * FRAME * CHANNELS
    times = []
    for i in range(args.warmup + args.steps):
        te = O.time_encode(sample, CHANNELS)
        td = O.time_decode(descs, words, CHANNELS)
        if i >= args.warmup:
            times.append((te, td))
    tot = [a + b for a, b in times]
    mean_s = statistics.fmean(tot)
    value = n_samples / mean_s / 1e6
    info = {
        "value": value, "unit": "MSamples/s", "cores": O.cores, "threads": O.cores, "kind": O.kind,
        "sample": "each step: first %d of %d frames (%.1f s of audio) encoded then decoded; timed: %s" % (
            sample_frames, n_frames, sample_frames * FRAME / SAMPLE_RATE,
            "sela::Encoder/Decoder::processFrames only" if O.kind == "reference" else "oracle port batch calls"),
        "encode_msamples_s": n_samples / statistics.fmean(t[0] for t in times) / 1e6,
        "decode_msamples_s": n_samples / statistics.fmean(t[1] for t in times) / 1e6,
        "step_ms_min": min(tot) * 1e3, "step_ms_max": max(tot) * 1e3,
        "whole_file_equivalent_ms": n_samples_file / (value * 1e6) * 1e3,
    }
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "MSamples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": mean_s * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64+int64", "data": "synthetic",
        "config": workload_config(n_frames, n_samples_file),
        "step_sample_frames": sample_frames,
        "cpu_baseline": info,
        "e2e": {"value": value, "unit": "MSamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit_line(line)


def run_ours(args, rank, world, local_rank):
    import torch
    import sela_b200
    from sela_b200 import _lib
    from sela_b200.device import DeviceCodec

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this implementation has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        # rank 0's stdout must carry exactly ONE line (the JSON), but NCCL writes its version banner
        # to fd 1 when the first communicator comes up: park the real stdout and point fd 1 at stderr
        # until the line is ready (emit_line)
        sys.stdout.flush()
        _REAL_STDOUT.append(os.dup(1))
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)

    sampler = ClockSampler(local_rank) if rank == 0 else None   # started early: nvidia-smi is slow to spin up
    pcm_np = make_pcm(1 + rank)
    n_frames = pcm_np.shape[0] // FRAME
    n_samples = n_frames * FRAME * CHANNELS
    L = _lib.lib()
    _lib.init(local_rank)

    # ---------------- device-resident leg ----------------
    pcm = torch.from_numpy(pcm_np.reshape(-1)).to(dev)
    out = torch.empty_like(pcm)
    codec = DeviceCodec(n_frames, CHANNELS, device=local_rank)
    codec.encode(pcm)
    torch.cuda.synchronize()
    codec.check_status()
    n_words = int(codec.words_used.item())
    codec.decode(out, n_words)
    torch.cuda.synchronize()
    codec.check_status()
    round_trip_ok = bool(torch.equal(out, pcm))

    def step():
        codec.encode(pcm)
        codec.decode(out, n_words)

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * args.steps + 1)]
    launches0 = L.selab200_launch_count()
    torch.cuda.synchronize()
    t_wall0 = time.time()
    ev[0].record()
    for i in range(args.steps):
        codec.encode(pcm)
        ev[2 * i + 1].record()
        codec.decode(out, n_words)
        ev[2 * i + 2].record()
    torch.cuda.synchronize()
    t_wall1 = time.time()
    if dist:
        dist.barrier()
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    launches = L.selab200_launch_count() - launches0
    total_ms = ev[0].elapsed_time(ev[-1])
    enc_ms = statistics.fmean(ev[2 * i].elapsed_time(ev[2 * i + 1]) for i in range(args.steps))
    dec_ms = statistics.fmean(ev[2 * i + 1].elapsed_time(ev[2 * i + 2]) for i in range(args.steps))
    codec.check_status()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, codec.descs.cpu().numpy().view(_lib.DESC_DTYPE),
                     codec.words[:int(codec.words_used.item())].cpu().numpy().view(np.uint32), out.cpu().numpy())

    # ---------------- end-to-end leg (host buffers through the public C ABI) ----------------
    def pinned(nbytes, dtype):
        p = L.selab200_host_alloc(nbytes)
        return np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(p)).view(dtype), p

    h_pcm, p1 = pinned(n_samples * 2, np.int16)
    h_pcm[:] = pcm_np.reshape(-1)
    h_out, p2 = pinned(n_samples * 2, np.int16)
    cap = L.selab200_encode_words_bound(n_frames, CHANNELS)
    h_words, p3 = pinned(cap * 4, np.uint32)
    h_descs, p4 = pinned(n_frames * CHANNELS * 32, np.uint8)
    used = C.c_size_t(0)

    split = [0.0, 0.0]   # seconds inside the encode call / the decode call (both synchronous)

    def e2e_step():
        t_a = time.perf_counter()
        _lib.check(L.selab200_encode_frames(h_pcm.ctypes.data, n_frames, CHANNELS, h_descs.ctypes.data,
                                            h_words.ctypes.data, cap, C.addressof(used)))
        t_b = time.perf_counter()
        _lib.check(L.selab200_decode_frames(h_descs.ctypes.data, n_frames, CHANNELS, h_words.ctypes.data,
                                            used.value, h_out.ctypes.data))
        split[0] += t_b - t_a
        split[1] += time.perf_counter() - t_b

    e2e_steps = args.steps
    for _ in range(3):
        e2e_step()
    if dist:
        dist.barrier()
    split[0] = split[1] = 0.0
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    e2e_ok = bool(np.array_equal(h_out, h_pcm))
    h2d = n_samples * 2 + n_frames * CHANNELS * 32 + used.value * 4      # PCM in; descs + words back in for decode
    d2h = n_frames * CHANNELS * 32 + used.value * 4 + n_samples * 2 + 16  # descs + words out; PCM out; status

    # ---------------- reductions ----------------
    t = torch.tensor([total_ms, e2e_s * 1e3], dtype=torch.float64, device=dev)
    if dist:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms_max, e2e_ms_max = t.tolist()
    total_samples = n_samples * world
    value = total_samples * args.steps / (total_ms_max * 1e-3) / 1e6
    e2e_value = total_samples / (e2e_ms_max * 1e-3) / 1e6

    # ---------------- the Rice-decode kernel on its own; PCIe rates of this box; the sharded configs ----------------
    peak, peak_src = measured_peak_hbm()
    rice = pcie = None
    if rank == 0:
        try:
            rice = rice_decode_roofline(codec, n_frames, n_words, dev, peak)
        except Exception as e:                      # never lose the headline to a side measurement
            rice = {"error": repr(e)[:300]}
        try:
            pcie = pcie_probe(dev)
        except Exception as e:
            pcie = {"error": repr(e)[:300]}
    line = None
    if rank == 0:
        desc_bytes = n_frames * CHANNELS * 32
        prof, stale = measured_profile("k_encode_units<stereo>")
        enc_bytes = n_samples * 2 + n_words * 4 + desc_bytes              # algorithmic: PCM in, words + descs out
        achieved = enc_bytes / (enc_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": "MSamples/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": total_ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64+int64",
            "data": "synthetic",
            "config": workload_config(n_frames, n_samples),
            "bits_per_sample": n_words * 32 / n_samples,
            "encode_msamples_s": n_samples / (enc_ms * 1e-3) / 1e6,
            "decode_msamples_s": n_samples / (dec_ms * 1e-3) / 1e6,
            "encode_ms": enc_ms, "decode_ms": dec_ms,
            "round_trip_bit_exact": round_trip_ok and e2e_ok,
            "e2e": {"value": e2e_value, "unit": "MSamples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms_max, "steps": e2e_steps,
                    "encode_ms": split[0] / e2e_steps * 1e3, "decode_ms": split[1] / e2e_steps * 1e3,
                    "pcie_probe": pcie,
                    "copy_floor_ms": None if not pcie or "error" in pcie else
                    (max(n_samples * 2 / pcie["h2d_gbs"], (used.value * 4 + n_frames * CHANNELS * 32) / pcie["d2h_gbs"]) +
                     max((used.value * 4 + n_frames * CHANNELS * 32) / pcie["h2d_gbs"], n_samples * 2 / pcie["d2h_gbs"])) / 1e6,
                    "note": "copy_floor_ms: the two calls of a step run one after the other and each overlaps its own upload and "
                            "download, so a step cannot beat max(PCM up, words down) + max(words up, PCM down) at the one-direction rates; "
                            "pcie_probe.*_both_directions = each direction's rate while the other is busy, which is what the "
                            "pipelined calls see most of the time"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"kernel": "k_encode_units<stereo> (fused analysis+FIR+Rice; + scan + gather launches)", "bound": "hbm",
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": (prof or {}).get("traffic"), "traffic_stale": stale, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": enc_bytes,
                         "compute": {"pipe": "fp64", "busy_frac": (prof or {}).get("fp64_busy_frac"),
                                     "issue_active_frac": (prof or {}).get("issue_active_frac"),
                                     "fp64_ops_per_launch": n_frames * 3 * (2 * FRAME * 101 + 2 * FRAME),
                                     "note": "busy_frac / issue_active_frac from the committed ncu capture (profiles/traffic.json); "
                                             "ops = sequentially rounded multiplies and adds of the 101-lag autocorrelation + mean, 3 units per stereo frame"},
                         "note": "FP64-latency / instruction-issue bound, not HBM bound (DESIGN.md 4); traffic = dram "
                                 "read+write per launch from profiles/traffic.json (ncu), traffic_stale = kernel sources "
                                 "changed since that capture"},
            "roofline_rice_decode": rice,
        }
        if world == 1 and not args.no_cpu:
            info, (sf, d_ref, w_ref) = cpu_reference_leg(pcm_np)
            line["cpu_baseline"] = info
            # bit-exactness against the CPU coder on the sampled frames
            descs_gpu = codec.descs.cpu().numpy().view(_lib.DESC_DTYPE)[: sf * CHANNELS]
            words_gpu = codec.words[: int(descs_gpu[-1]["res_offset"]) + int(descs_gpu[-1]["res_words"])].cpu().numpy().view(np.uint32)
            line["bit_exact_vs_cpu"] = bool(descs_gpu.tobytes() == d_ref.tobytes() and np.array_equal(words_gpu, w_ref))

    # ---------------- configs[3] / [4]: one file across the ranks, a batch of files per rank ----------------
    # The headline above is complete at this point.  The sharded block runs collectives of its own; should a
    # rank fail or stall in it, a watchdog lets rank 0 print the line without it instead of losing the run.
    if not args.no_sharded:
        import threading
        done = threading.Event()

        def watchdog():
            if not done.wait(args.sharded_timeout):
                if rank == 0:
                    line["sharded"] = {"error": "sharded block did not finish within %d s" % args.sharded_timeout}
                    emit_line(line)
                os._exit(0)
        if dist:
            threading.Thread(target=watchdog, daemon=True).start()
        del pcm, out
        torch.cuda.empty_cache()
        try:
            sharded = sharded_block(args, rank, world, dev, dist)
        except Exception as e:
            sharded = {"error": repr(e)[:400]}
            if dist:                                 # the other ranks may be waiting for this one: do not join them again
                if rank == 0:
                    line["sharded"] = sharded
                    emit_line(line)
                done.set()
                os._exit(0)
        done.set()
        if rank == 0:
            line["sharded"] = sharded
    if rank == 0:
        emit_line(line)
    for p in (p1, p2, p3, p4):
        L.selab200_host_free(p)
    if dist:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--no-sharded", action="store_true", help="skip the configs[3]/[4] block (profiling runs)")
    ap.add_argument("--sharded-minutes", type=int, default=0, help="length of the config-4 file (default 60)")
    ap.add_argument("--sharded-timeout", type=int, default=240, help="seconds before the sharded block is given up (N > 1)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm codes a sample sized by a timing probe, not a fixed input")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
