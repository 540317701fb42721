"""The C++ mirror of the reference interface and the CLI built on it (sela_b200/host).

CPU part: the container code (WAV / .sela readers and writers) against the reference's file code.
GPU part: `sela -e/-d` byte-for-byte against the reference CLI, the reference's own main.cpp linked
against this library, and the reference's unit tests re-expressed on the mirror classes.
Digests of what the reference CLI wrote for the WAVs of _cases() (the .sela, and the .wav it decodes that
to) are stored in tests/golden/reference_cli.npz by tests/golden/make_golden.py."""
import pathlib
import struct
import subprocess

import numpy as np
import pytest

import oracle_lib as ol
from sela_b200 import synth, wavio

ROOT = pathlib.Path(__file__).resolve().parent.parent
BIN = ROOT / "sela_b200" / "host" / "bin"


def _run(*cmd, ok=True, env=None):
    import os
    p = subprocess.run([str(c) for c in cmd], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, **env) if env else None)
    if ok:
        assert p.returncode == 0, (cmd, p.stdout[-400:], p.stderr[-400:])
    return p


def _ensure_built():
    if not (BIN / "sela").exists():
        subprocess.run(["make", "-C", str(ROOT / "sela_b200" / "host")], check=True, capture_output=True)


def _cases(tmp):
    out = {}
    pcm = synth.sine_noise(44100, 2, n_frames=20, seed=1)
    pcm[2048 * 4:2048 * 9, 1] = pcm[2048 * 4:2048 * 9, 0] - (pcm[2048 * 4:2048 * 9, 1] >> 5)
    pcm = np.concatenate([pcm, pcm[:777]])                       # tail that is not a whole frame: dropped
    wavio.write_wav(tmp / "stereo.wav", pcm, 44100, extra_chunks=[(b"LIST", b"INFOabcd1234")])
    out["stereo"] = tmp / "stereo.wav"
    wavio.write_wav(tmp / "mono.wav", synth.sine_noise(22050, 1, n_frames=7, seed=5), 22050)
    out["mono"] = tmp / "mono.wav"
    wavio.write_wav(tmp / "oct.wav", synth.sine_noise(48000, 8, n_frames=5, seed=2), 48000)
    out["oct"] = tmp / "oct.wav"
    return out


def _file_digest(path):
    return ol.digest(np.frombuffer(path.read_bytes(), np.uint8))


def _reference_sela(name, wav):
    """The .sela bytes the reference CLI writes for `wav`: the CPU oracle's frames in the reference's file layout,
    checked against the digest of what the reference wrote."""
    raw = wav.read_bytes()
    ch, rate = struct.unpack_from("<HI", raw, 22)
    pcm = np.frombuffer(raw, "<i2", offset=raw.index(b"data") + 8)
    pcm = pcm[: pcm.size // (2048 * ch) * 2048 * ch]                 # the reference drops the partial last frame
    blob = wavio.pack_container(*ol.load("port").encode_frames(pcm, ch), rate, ch)
    assert ol.digest(np.frombuffer(blob, np.uint8)) == ol.golden("reference_cli")[name + "_sela"], name
    return blob


# ------------------------------------------------------------------ CPU --

def test_container_code_matches_reference(tmp_path):
    """file::SelaFile read->write is byte-identical on reference-produced files; file::WavFile
    read->(canonical)write equals what the reference decoder writes back (header + tail drop)."""
    _ensure_built()
    ref = ol.golden("reference_cli")
    for name, wav in _cases(tmp_path).items():
        ref_sela = tmp_path / (name + ".ref.sela")
        ref_sela.write_bytes(_reference_sela(name, wav))
        _run(BIN / "container_check", "sela", ref_sela, tmp_path / "rt.sela")
        assert (tmp_path / "rt.sela").read_bytes() == ref_sela.read_bytes(), name
        _run(BIN / "container_check", "wav", wav, tmp_path / "rt.wav")
        assert _file_digest(tmp_path / "rt.wav") == ref[name + "_wav"], name


def test_container_errors_match_reference_messages(tmp_path):
    _ensure_built()
    (tmp_path / "tiny.wav").write_bytes(b"RIFF")
    p = _run(BIN / "container_check", "wav", tmp_path / "tiny.wav", tmp_path / "o", ok=False)
    assert p.returncode == 1 and "File is too small, probably not a wav file." in p.stderr
    (tmp_path / "bad.sela").write_bytes(b"NotSela" + bytes(20))
    p = _run(BIN / "container_check", "sela", tmp_path / "bad.sela", tmp_path / "o", ok=False)
    assert p.returncode == 1 and "Magic number is incorrect" in p.stderr
    pcm8 = np.zeros((4096, 1), np.int16)
    wavio.write_wav(tmp_path / "w.wav", pcm8, 8000)
    raw = bytearray((tmp_path / "w.wav").read_bytes())
    raw[34] = 24                                                   # bitsPerSample = 24
    (tmp_path / "w24.wav").write_bytes(bytes(raw))
    p = _run(BIN / "container_check", "wav", tmp_path / "w24.wav", tmp_path / "o", ok=False)
    assert p.returncode == 1 and "Only 16bits per sample wav is supported." in p.stderr


# ------------------------------------------------------------------ GPU --

@pytest.mark.gpu
def test_reference_unit_tests_on_mirror_classes():
    _ensure_built()
    p = _run(BIN / "sela_reftests")
    assert "All tests passed" in p.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("binary", ["sela", "sela-classic", "sela_refmain"])
def test_cli_byte_parity_with_reference_cli(tmp_path, binary):
    """`sela`: the fused file-to-file drivers (Encoder/Decoder::processTo over the container entry
    points); `sela-classic`: the same binary on the reference's two-step call sequence;
    `sela_refmain`: the reference's own main.cpp compiled unchanged over the mirror classes."""
    _ensure_built()
    env = {"SELA_B200_CLASSIC": "1"} if binary == "sela-classic" else None
    binary = binary.split("-")[0]
    if not (BIN / binary).exists():
        pytest.skip("%s not built (needs the reference tree at build time)" % binary)
    ref = ol.golden("reference_cli")
    for name, wav in _cases(tmp_path).items():
        ours_sela, ours_wav = tmp_path / (name + ".sela"), tmp_path / (name + ".out.wav")
        p = _run(BIN / binary, "-e", wav, ours_sela, env=env)
        assert "Encoding: " in p.stdout
        _run(BIN / binary, "-d", ours_sela, ours_wav, env=env)
        assert _file_digest(ours_sela) == ref[name + "_sela"], name                # bit-identical .sela
        assert _file_digest(ours_wav) == ref[name + "_wav"], name                 # bit-identical .wav
        # lossless against the source (whole frames only)
        _, ch, pcm_out = wavio.read_wav_pcm(ours_wav)
        data_at = wav.read_bytes().index(b"data") + 8
        pcm_src = np.frombuffer(wav.read_bytes()[data_at:], dtype="<i2")
        pcm_src = pcm_src[: (pcm_src.size // (2048 * ch)) * 2048 * ch].reshape(-1, ch)
        assert np.array_equal(pcm_out, pcm_src), name


@pytest.mark.gpu
def test_cli_error_convention(tmp_path):
    _ensure_built()
    (tmp_path / "junk.wav").write_bytes(b"not a wav file at all, but long enough to pass the size check....")
    p = _run(BIN / "sela", "-e", tmp_path / "junk.wav", tmp_path / "o.sela", ok=False)
    assert p.returncode == 1 and "chunkId is not RIFF" in p.stderr
    p = _run(BIN / "sela", ok=True)
    assert "Usage:" in p.stdout
    # decode side: the reader's messages, on both call sequences
    wavio.write_wav(tmp_path / "a.wav", synth.sine_noise(8000, 1, n_frames=3, seed=1), 8000)
    _run(BIN / "sela", "-e", tmp_path / "a.wav", tmp_path / "a.sela")
    blob = (tmp_path / "a.sela").read_bytes()
    (tmp_path / "cut.sela").write_bytes(blob[:-9])
    (tmp_path / "magic.sela").write_bytes(b"SeLb" + blob[4:])
    (tmp_path / "tiny.sela").write_bytes(blob[:10])
    for env in (None, {"SELA_B200_CLASSIC": "1"}):
        for name, msg in (("cut", "sela file is truncated"), ("magic", "Magic number is incorrect"),
                          ("tiny", "File is too small, probably not a sela file.")):
            p = _run(BIN / "sela", "-d", tmp_path / (name + ".sela"), tmp_path / "o.wav", ok=False, env=env)
            assert p.returncode == 1 and msg in p.stderr, (name, env, p.stderr)
    # an empty WAV (no whole frame) encodes to the bare header and decodes to a bare WAV header
    wavio.write_wav(tmp_path / "short.wav", np.zeros((100, 2), np.int16), 44100)
    outs = []
    for env in (None, {"SELA_B200_CLASSIC": "1"}):
        _run(BIN / "sela", "-e", tmp_path / "short.wav", tmp_path / "short.sela", env=env)
        _run(BIN / "sela", "-d", tmp_path / "short.sela", tmp_path / "short.out.wav", env=env)
        outs.append(((tmp_path / "short.sela").read_bytes(), (tmp_path / "short.out.wav").read_bytes()))
    assert outs[0] == outs[1] and len(outs[0][0]) == 15 and len(outs[0][1]) == 44


@pytest.mark.gpu
def test_cli_batch_mode_equals_one_file_at_a_time(tmp_path):
    """`sela -E/-D out_dir files...`: many files in one process (pinned staging reused per worker thread,
    files on the GPU one after the other).  Same bytes as one process per file; a bad file is reported
    and does not stop the rest."""
    _ensure_built()
    cases = _cases(tmp_path)
    for i in range(6):   # enough files that every worker thread reuses its staging buffers
        wavio.write_wav(tmp_path / ("s%d.wav" % i), synth.sine_noise(44100, 2, n_frames=3 + 2 * i, seed=40 + i), 44100)
        cases["s%d" % i] = tmp_path / ("s%d.wav" % i)
    (tmp_path / "junk.wav").write_bytes(b"not a wav file at all, but long enough to pass the size check....")
    enc, dec = tmp_path / "enc", tmp_path / "dec"
    enc.mkdir()
    dec.mkdir()
    wavs = [cases[k] for k in sorted(cases)]
    p = _run(BIN / "sela", "-E", enc, *wavs, tmp_path / "junk.wav", ok=False, env={"SELA_B200_WORKERS": "3"})
    assert p.returncode == 1 and "junk.wav: chunkId is not RIFF" in p.stderr, (p.stdout, p.stderr)
    assert "Encoded %d of %d files" % (len(wavs), len(wavs) + 1) in p.stdout
    p = _run(BIN / "sela", "-D", dec, *[enc / (w.stem + ".sela") for w in wavs], env={"SELA_B200_WORKERS": "3"})
    assert "Decoded %d of %d files" % (len(wavs), len(wavs)) in p.stdout
    for w in wavs:
        _run(BIN / "sela", "-e", w, tmp_path / "one.sela")
        _run(BIN / "sela", "-d", tmp_path / "one.sela", tmp_path / "one.wav")
        assert (enc / (w.stem + ".sela")).read_bytes() == (tmp_path / "one.sela").read_bytes(), w.name
        assert (dec / (w.stem + ".wav")).read_bytes() == (tmp_path / "one.wav").read_bytes(), w.name
