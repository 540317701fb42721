#!/usr/bin/env python3
"""Generate the golden vectors under tests/golden/ from the UNMODIFIED reference.

    python tests/golden/make_golden.py <reference checkout> [frames] [stages] [cli]

builds oracle/_ref from that checkout (oracle/Makefile) and writes the files named (default: all).
The reference ships no golden files (SURVEY.md 4), so these are outputs of the reference's own
classes (through oracle/ref_shim.cpp) and CLI (oracle/ref_cli_main.cpp) on seeded inputs.
They let the tests compare with the reference on machines that do not have it.

  golden_frames.npz
    pcm_<case>      int16 [n_frames*2048, channels]   input
    descs_<case>    structured (32-byte descriptor)   reference encoder output
    words_<case>    uint32                            reference encoder output (arena)
    decoded_<case>  int16                             reference DECODER output for (descs, words)

  reference_stages.npz   (tests/test_oracle_vs_ref.py, tests/test_host_logic.py)
    fam_<name>_*           LPC analysis, Rice streams and decodes of signals.families()
    rand_*, dc_*           order / coefficients / residue digest of signals.random_frames(300, 11), DC frames
    rice_<i>_*             Rice parameter, words and decode of test_oracle_vs_ref.rice_inputs()
    batch<ch>_*            descriptors, word digest and decode digest of test_oracle_vs_ref.batch_pcm(ch)
    lpc_first_order_bits   uint64[128]: the reference's firstOrderCoefficients as IEEE-754 bit patterns

  reference_cli.npz      (tests/test_host_cli.py, tests/test_container.py, tests/test_multi_device.py)
    <case>_sela, _wav      digests of what the reference CLI's -e wrote for test_host_cli._cases(), and of
                           what its -d wrote for that .sela
    pack_<ch>_sela         digest of its -e output for test_container.pack_cases()
    oct700_sela, _wav      digests of its -e / -d output for the 700-frame 8-channel WAV

Digests are oracle_lib.digest (SHA-256 over dtype and bytes, 128 bits): they stand for outputs too
large to keep, so a mismatch says only that the bytes differ.
"""
import pathlib
import re
import struct
import subprocess
import sys
import tempfile

import numpy as np

HERE = pathlib.Path(__file__).resolve().parent
ROOT = HERE.parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

import oracle_lib as ol  # noqa: E402
import signals  # noqa: E402
from sela_b200 import synth, wavio  # noqa: E402


def cases():
    out = {}
    st = synth.sine_noise(44100, 2, n_frames=6, seed=1)                       # BASELINE config 2/3 shape
    st[2048 * 2:2048 * 4, 1] = st[2048 * 2:2048 * 4, 0] - (st[2048 * 2:2048 * 4, 1] >> 5)
    st[2048 * 4:2048 * 5, 1] = st[2048 * 4:2048 * 5, 0]
    out["stereo"] = st
    out["mono_config1"] = synth.config1_frame().astype(np.int16).reshape(-1, 1)  # BASELINE config 1
    out["oct"] = synth.sine_noise(48000, 8, n_frames=2, seed=2)                # config 4 shape
    fam = signals.families()
    names = sorted(fam)
    out["edge_mono"] = np.concatenate([fam[n] for n in names]).astype(np.int16).reshape(-1, 1)
    out["edge_stereo"] = np.concatenate(
        [np.stack([fam[n], fam[names[(i * 5 + 2) % len(names)]]], axis=1) for i, n in enumerate(names)]).astype(np.int16)
    out["three"] = synth.sine_noise(32000, 3, n_frames=2, seed=9)
    # Two frames of the config-4-shaped 10-minute file (48 kHz, 8 channels, seed 2) on which the REFERENCE is
    # not lossless: its decoder departs from the source at sample 1 of one channel (frame 8975 channel 1,
    # frame 13577 channel 4; encoder and decoder round the prediction differently when the Q35 sum lands
    # exactly on a half, SURVEY.md 7.3).  The decoded_* array pins what the reference decoder returns.
    big = synth.sine_noise(48000, 8, 600, seed=2)
    out["oct_reference_lossy"] = np.concatenate([big[8975 * 2048:8976 * 2048], big[13577 * 2048:13578 * 2048]])
    return out


def frames(R):
    blob = {}
    for name, pcm in cases().items():
        ch = pcm.shape[1]
        descs, words = R.encode_frames(pcm, ch)
        blob["pcm_" + name] = pcm
        blob["descs_" + name] = descs
        blob["words_" + name] = words
        blob["decoded_" + name] = R.decode_frames(descs, words, ch)
        print("%-14s ch=%d frames=%d words=%d lossless=%s" % (
            name, ch, pcm.shape[0] // 2048, words.size, np.array_equal(blob["decoded_" + name], pcm.reshape(-1))))
    return blob


def _padded_q(q):
    out = np.zeros(100, np.int32)
    out[:q.size] = q
    return out


def stages(R, ref_tree):
    import test_oracle_vs_ref as t
    blob = {}
    for name, s in signals.families().items():
        a = R.lpc_analyse(s)
        kq, wq = R.rice_encode(a["q"])
        kr, wr = R.rice_encode(a["res"])
        p = "fam_%s_" % name
        blob.update({p + "order": a["order"], p + "q": a["q"], p + "c": a["c"], p + "res": a["res"],
                     p + "kq": kq, p + "wq": wq, p + "kr": kr, p + "wr": wr,
                     p + "decoded_q": ol.digest(R.rice_decode(wq, kq, a["q"].size)),
                     p + "decoded_r": ol.digest(R.rice_decode(wr, kr, a["res"].size)),
                     p + "synthesised": ol.digest(R.lpc_synthesise(a["res"], a["order"], a["q"]))})
    for key, frames_ in (("rand", signals.random_frames(300, seed=11)),
                         ("dc", [np.full(2048, v, np.int32) for v in t.dc_levels()])):
        an = [R.lpc_analyse(s) for s in frames_]
        blob[key + "_order"] = np.array([a["order"] for a in an], np.int32)
        blob[key + "_q"] = np.stack([_padded_q(a["q"]) for a in an])
        blob[key + "_res"] = np.array([ol.digest(a["res"]) for a in an])
    blob["dc_level"] = np.array(t.dc_levels(), np.int32)
    for i, x in enumerate(t.rice_inputs()):
        k, w = R.rice_encode(x)
        blob["rice_%d_k" % i], blob["rice_%d_words" % i] = k, w
        blob["rice_%d_decoded" % i] = ol.digest(R.rice_decode(w, k, x.size))
    for ch in (1, 2, 3, 8):
        d, w = R.encode_frames(t.batch_pcm(ch), ch)
        blob["batch%d_descs" % ch], blob["batch%d_words" % ch] = d, ol.digest(w)
        blob["batch%d_decoded" % ch] = ol.digest(R.decode_frames(d, w, ch))
    text = (ref_tree / "src" / "include" / "lpc.hpp").read_text()
    m = re.search(r"firstOrderCoefficients\[128\]\s*=\s*\{([^}]*)\}", text)
    vals = [float(v) for v in m.group(1).replace("\n", " ").split(",") if v.strip()]
    assert len(vals) == 128
    blob["lpc_first_order_bits"] = np.array([struct.unpack("<Q", struct.pack("<d", v))[0] for v in vals], np.uint64)
    return blob


def cli():
    import test_container
    import test_host_cli
    exe = ROOT / "oracle" / "_ref" / "sela_ref_cli"
    file_digest = lambda p: ol.digest(np.frombuffer(p.read_bytes(), np.uint8))

    def run(mode, src, dst):
        subprocess.run([str(exe), mode, str(src), str(dst)], check=True, capture_output=True, timeout=600)

    blob = {}
    with tempfile.TemporaryDirectory() as tmp:
        tmp = pathlib.Path(tmp)
        for name, wav in test_host_cli._cases(tmp).items():
            run("-e", wav, tmp / "r.sela")
            run("-d", tmp / "r.sela", tmp / "r.wav")
            blob[name + "_sela"] = file_digest(tmp / "r.sela")
            blob[name + "_wav"] = file_digest(tmp / "r.wav")
        for ch, rate, pcm in test_container.pack_cases():
            wavio.write_wav(tmp / "in.wav", pcm, rate)
            run("-e", tmp / "in.wav", tmp / "r.sela")
            blob["pack_%d_sela" % ch] = file_digest(tmp / "r.sela")
        wavio.write_wav(tmp / "oct.wav", synth.sine_noise(48000, 8, n_frames=700, seed=2), 48000)
        run("-e", tmp / "oct.wav", tmp / "r.sela")
        run("-d", tmp / "r.sela", tmp / "r.wav")
        blob["oct700_sela"], blob["oct700_wav"] = file_digest(tmp / "r.sela"), file_digest(tmp / "r.wav")
    return blob


def main():
    ref_tree = pathlib.Path(sys.argv[1]).resolve()
    which = sys.argv[2:] or ["frames", "stages", "cli"]
    subprocess.run(["make", "-C", str(ROOT / "oracle"), "SELA_REF=%s" % ref_tree], check=True, capture_output=True)
    R = ol.load("ref")
    assert R.kind == "reference"
    if "frames" in which:
        np.savez_compressed(HERE / "golden_frames.npz", **frames(R))
    if "stages" in which:
        np.savez_compressed(HERE / "reference_stages.npz", **stages(R, ref_tree))
    if "cli" in which:
        np.savez_compressed(HERE / "reference_cli.npz", **cli())


if __name__ == "__main__":
    main()
