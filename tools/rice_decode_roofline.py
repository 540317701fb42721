"""The Rice-decode kernel (K5) in isolation against the HBM roofline, as a function of batch size.

north_star asks for ">= 70 % of HBM roofline on the Rice decode kernel".  The kernel is one lane per
stream; at BASELINE's batch (25 838 streams = 808 warps) it is starved for parallelism.  This sweeps
the number of streams by tiling the coded 10-minute stereo file.
Algorithmic bytes (SURVEY.md 8d): residue words read + 4 B per decoded sample written.
Run on the GPU box:  python tools/rice_decode_roofline.py [max_tile]
"""
import ctypes as C, json, os, sys
import numpy as np, torch
sys.path.insert(0, ".")
from sela_b200 import _lib, synth
from sela_b200.device import DeviceCodec

PEAK = json.load(open("MEASURED_PEAKS.json"))["hbm_gbs"] if os.path.exists("MEASURED_PEAKS.json") else 6650.0
import argparse
ap = argparse.ArgumentParser()
ap.add_argument("max_tile", nargs="?", type=int, default=48)
ap.add_argument("--tiles", default="1,4,16,48,96")
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--warm", type=int, default=3)
ap.add_argument("--out", default="gpurun_out/rice_decode_roofline.json")
ap.add_argument("--frames", type=int, default=0, help="use only the first N frames of the file (small-batch sweep)")
ap.add_argument("--splits", default="auto", help="comma list of SELAB200_RICE_SPLIT values (auto = library default)")
args = ap.parse_args()
max_tile = args.max_tile
TILES = [int(t) for t in args.tiles.split(",")]
pcm = synth.sine_noise(44100, 2, seconds=600, seed=1)
if args.frames:
    pcm = pcm[: args.frames * 2048]
n_frames = pcm.shape[0] // 2048
codec = DeviceCodec(n_frames, 2)
codec.encode(torch.from_numpy(pcm.reshape(-1)).cuda()); torch.cuda.synchronize(); codec.check_status()
n_words = int(codec.words_used.item())
descs = codec.descs.cpu().numpy().view(_lib.DESC_DTYPE).copy()
words = codec.words[:n_words].clone()
res_words = int(descs["res_words"].astype(np.int64).sum())
L = _lib.lib()
rows = []
ref_out = None
for tile in [t for t in TILES if t <= max_tile]:
    d = np.tile(descs, tile)
    for r in range(tile):
        sl = slice(r * descs.size, (r + 1) * descs.size)
        d["refl_offset"][sl] += r * n_words
        d["res_offset"][sl] += r * n_words
    d_descs = torch.from_numpy(d.view(np.uint8).reshape(-1)).cuda()
    d_words = words.repeat(tile)
    n_sub = d.size
    out = torch.empty(n_sub * 2048, dtype=torch.int32, device="cuda")
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    for split in args.splits.split(","):
        ring = split
        if split == "auto":
            os.environ.pop("SELAB200_RICE_SPLIT", None)
        else:
            os.environ["SELAB200_RICE_SPLIT"] = split
        def run():
            _lib.check(L.selab200_rice_decode_frames_device(d_descs.data_ptr(), n_frames * tile, 2, d_words.data_ptr(),
                                                            n_words * tile, out.data_ptr(), status.data_ptr(), C.c_void_p(stream)))
        for _ in range(args.warm):
            run()
        torch.cuda.synchronize()
        assert int(status.item()) == 0
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        reps = args.reps
        ev[0].record()
        for _ in range(reps):
            run()
        ev[1].record(); torch.cuda.synchronize()
        ms = ev[0].elapsed_time(ev[1]) / reps
        samples = n_sub * 2048
        alg = res_words * tile * 4 + samples * 4
        gbs = alg / ms / 1e6
        flagged = C.c_uint32(0)
        _lib.check(L.selab200_rice_decode_flagged(C.addressof(flagged)))
        if ref_out is None:
            ref_out = out[: descs.size * 2048].clone()      # first configuration of the first tile
        same = bool(torch.equal(out[: descs.size * 2048], ref_out))
        rows.append(dict(streams=n_sub, split=split, ms=ms, gsamples_s=samples / ms / 1e6, gb_s=gbs, frac_of_hbm_peak=gbs / PEAK,
                         flagged=flagged.value, algorithmic_bytes=alg, same_as_first=same))
        print("streams %8d  split %4s  %8.3f ms  %7.1f GSamples/s  %7.1f GB/s  = %.1f %% of measured HBM peak (%.0f GB/s)  flagged %d  same %s" % (
            n_sub, split, ms, samples / ms / 1e6, gbs, 100 * gbs / PEAK, PEAK, flagged.value, same))
    if tile > 1:  # every tile must decode to the same residues as the first
        a = out[: descs.size * 2048]
        assert torch.equal(out[-descs.size * 2048:], a)
    del out, d_words, d_descs
os.makedirs("gpurun_out", exist_ok=True)
json.dump(rows, open(args.out, "w"), indent=1)
