"""The byte-packed .sela container (SURVEY.md 8f, row f2): host-only frame walk, and the
device paths that write / read whole containers (selab200_encode_container,
selab200_container_open / _decode).  Reference: src/file/sela_file.cpp:19-137."""
import pathlib
import struct
import subprocess

import numpy as np
import pytest

import oracle_lib as ol
from sela_b200 import SelaB200Error, codec, synth, wavio

ROOT = pathlib.Path(__file__).resolve().parent.parent
FRAME = 2048


@pytest.fixture(scope="module")
def O():
    return ol.best()


def _stereo(n_frames, seed):
    pcm = synth.sine_noise(44100, 2, n_frames=n_frames, seed=seed)
    if n_frames >= 6:
        pcm[FRAME * 2:FRAME * 5, 1] = pcm[FRAME * 2:FRAME * 5, 0] - (pcm[FRAME * 2:FRAME * 5, 1] >> 6)
    return pcm


def _blob(O, pcm, channels, rate=44100):
    d, w = O.encode_frames(pcm, channels)
    return wavio.pack_container(d, w, rate, channels), d, w


# ------------------------------------------------------------------ CPU --

def pack_cases():
    """(channels, rate, pcm) of the WAVs the reference CLI encoded for tests/golden/reference_cli.npz."""
    return [(channels, rate, _stereo(n, 4) if channels == 2 else synth.sine_noise(rate, channels, n_frames=n, seed=6))
            for channels, rate, n in ((2, 44100, 9), (1, 22050, 4), (8, 48000, 3))]


def test_pack_container_helper_equals_reference_writer(O):
    """Pins the test helper itself: oracle frames packed by wavio.pack_container are the bytes the
    reference CLI wrote for the same WAV."""
    for channels, rate, pcm in pack_cases():
        blob, _, _ = _blob(O, pcm, channels, rate)
        assert ol.digest(np.frombuffer(blob, np.uint8)) == ol.golden("reference_cli")["pack_%d_sela" % channels], channels


def test_container_walk_matches_descriptors(O):
    pcm = _stereo(11, 2)
    blob, d, w = _blob(O, pcm, 2)
    info = codec.container_info(blob)
    assert info == {"sample_rate": 44100, "bits_per_sample": 16, "channels": 2, "header_frames": 11,
                    "n_frames": 11, "n_words": w.size, "n_bytes_used": len(blob)}
    # trailing bytes after the last declared frame are never looked at
    assert codec.container_info(blob + b"\x00\xff\x55\xaa junk")["n_frames"] == 11
    # a header that promises more frames than the bytes hold: the walk stops at the end, quietly
    more = bytearray(blob)
    more[11:15] = struct.pack("<I", 500)
    assert codec.container_info(bytes(more))["n_frames"] == 11


def test_container_walk_stops_at_bad_sync_and_reports_truncation(O):
    pcm = _stereo(6, 3)
    blob, d, w = _blob(O, pcm, 2)
    # byte position of frame 4's sync word: header + 4 frames (sync + 2 x 12 header bytes) + their words
    words4 = int(d[8]["refl_offset"])
    at = 15 + 4 * (4 + 2 * 12) + 4 * words4
    assert blob[at:at + 4] == wavio.SELA_SYNC
    bad = bytearray(blob)
    bad[at + 1] ^= 0x40
    info = codec.container_info(bytes(bad))
    assert info["n_frames"] == 4 and info["n_words"] == words4 and info["n_bytes_used"] == at
    for cut in (1, 7, 640, len(blob) - 19, len(blob) - 27):
        with pytest.raises(SelaB200Error, match="sela file is truncated"):
            codec.container_info(blob[:len(blob) - cut])
    assert codec.container_info(blob[:15])["n_frames"] == 0          # header only: zero frames, no error
    assert codec.container_info(blob[:17])["n_frames"] == 0          # sync word cut short: quiet stop, like the reference
    with pytest.raises(SelaB200Error, match="File is too small"):
        codec.container_info(blob[:14])
    with pytest.raises(SelaB200Error, match="Magic number is incorrect"):
        codec.container_info(b"RIFF" + blob[4:])


# ------------------------------------------------------------------ GPU --

@pytest.mark.gpu
@pytest.mark.parametrize("channels,n_frames,rate", [(1, 9, 22050), (2, 24, 44100), (3, 5, 48000), (8, 4, 48000)])
def test_encode_container_is_the_reference_byte_stream(O, channels, n_frames, rate):
    pcm = _stereo(n_frames, 3) if channels == 2 else synth.sine_noise(rate, channels, n_frames=n_frames, seed=2)
    blob, _, _ = _blob(O, pcm, channels, rate)
    ours = codec.encode_container(pcm, channels, rate)
    assert ours.tobytes() == blob
    info, out = codec.decode_container(blob)
    assert (info["n_frames"], info["channels"], info["sample_rate"]) == (n_frames, channels, rate)
    assert np.array_equal(out, pcm.reshape(-1))


@pytest.mark.gpu
def test_container_paths_chunked(O, monkeypatch):
    """Many tiny pipeline chunks: chunk boundaries fall on arbitrary byte alignments."""
    pcm = _stereo(23, 8)
    blob, _, _ = _blob(O, pcm, 2)
    for cf in ("1", "3", "7"):
        monkeypatch.setenv("SELAB200_CHUNK_FRAMES", cf)
        assert codec.encode_container(pcm, 2, 44100).tobytes() == blob, cf
        assert np.array_equal(codec.decode_container(blob)[1], pcm.reshape(-1)), cf
    monkeypatch.delenv("SELAB200_CHUNK_FRAMES")


@pytest.mark.gpu
def test_container_word_alignment_cases(O):
    """Reflection-word counts 1..4 shift the residue words through all four byte alignments;
    mono frames put the next sync word at every alignment too."""
    rng = np.random.default_rng(12)
    frames = []
    for order_hint in (1, 6, 14, 30, 60, 100):
        t = np.arange(FRAME)
        x = sum(np.sin(2 * np.pi * (0.01 + 0.004 * h) * t + h) for h in range(order_hint)) / order_hint
        frames.append(np.clip(np.round(9000 * x + rng.normal(0, 3 + order_hint, FRAME)), -32768, 32767))
    pcm = np.concatenate(frames).astype(np.int16).reshape(-1, 1)
    blob, d, _ = _blob(O, pcm, 1, 8000)
    assert len(set(int(v) % 4 for v in d["refl_words"])) >= 2
    assert codec.encode_container(pcm, 1, 8000).tobytes() == blob
    assert np.array_equal(codec.decode_container(blob)[1], pcm.reshape(-1))


@pytest.mark.gpu
def test_decode_container_damaged_input(O):
    pcm = _stereo(6, 3)
    blob, d, w = _blob(O, pcm, 2)
    at = 15 + 4 * (4 + 2 * 12) + 4 * int(d[8]["refl_offset"])
    bad = bytearray(blob)
    bad[at] = 0x01                                             # frame 4's sync word
    info, out = codec.decode_container(bytes(bad))
    assert info["n_frames"] == 4 and np.array_equal(out, pcm.reshape(-1)[:4 * 2 * FRAME])
    with pytest.raises(SelaB200Error, match="sela file is truncated"):
        codec.decode_container(blob[:-5])
    info, out = codec.decode_container(blob[:15])
    assert info["n_frames"] == 0 and out.size == 0
    # a subframe header that fails validation (order 101) is refused on the device, not decoded
    bad = bytearray(blob)
    bad[15 + 4 + 6] = 101
    with pytest.raises(SelaB200Error) as e:
        codec.decode_container(bytes(bad))
    assert e.value.status == -6


@pytest.mark.gpu
def test_encode_container_capacity(O):
    pcm = _stereo(4, 1)
    blob, _, _ = _blob(O, pcm, 2)
    with pytest.raises(SelaB200Error) as e:
        codec.encode_container(pcm, 2, 44100, capacity=len(blob) - 4)
    assert e.value.status == -4
    with pytest.raises(SelaB200Error) as e:
        codec.encode_container(pcm, 2, 44100, capacity=40)
    assert e.value.status == -4
    assert codec.encode_container(pcm, 2, 44100, capacity=len(blob)).tobytes() == blob
    # zero frames: the 15-byte header alone
    empty = codec.encode_container(np.zeros(0, np.int16), 2, 8000)
    assert empty.tobytes() == b"SeLa" + struct.pack("<IHBI", 8000, 16, 2, 0)


@pytest.mark.gpu
def test_full_baseline_container_round_trip(O):
    """BASELINE configs[1]/[2] at full size through the container paths: the .sela bytes equal the
    CPU coder's frames in the reference file layout, and decode back to the source."""
    pcm = synth.sine_noise(44100, 2, seconds=600, seed=1)
    ours = codec.encode_container(pcm, 2, 44100)
    d_ref, w_ref = O.encode_frames(pcm, 2)
    assert ours.tobytes() == wavio.pack_container(d_ref, w_ref, 44100, 2)
    info, out = codec.decode_container(ours)
    assert info["n_frames"] == 12919 and np.array_equal(out, pcm.reshape(-1))


def test_walker_agrees_with_the_value_struct_reader_on_damaged_files(O, tmp_path):
    """Two parsers read .sela bytes: file::SelaFile::readFromFile of the C++ mirror (builds the
    reference's value structs) and the library's copy-free walk.  On truncated / corrupted input they
    must agree: same error message, or the same frames -- checked through the bytes the struct reader
    writes back (header + exactly the frames it accepted)."""
    host_bin = ROOT / "sela_b200" / "host" / "bin" / "container_check"
    if not host_bin.exists():
        subprocess.run(["make", "-C", str(ROOT / "sela_b200" / "host")], check=True, capture_output=True)
    pcm = _stereo(5, 7)
    blob, _, _ = _blob(O, pcm, 2)
    mono, _, _ = _blob(O, synth.sine_noise(8000, 1, n_frames=3, seed=9), 1, 8000)
    rng = np.random.default_rng(77)
    cases = []
    for base in (blob, mono):
        n = len(base)
        cases += [base[:c] for c in sorted(set(int(v) for v in rng.integers(0, n, 24)) | {0, 3, 14, 15, 16, 18, 19, 26, n - 1})]
        for _ in range(24):                     # one flipped byte: header fields, sync words, counts, payload
            b = bytearray(base)
            at = int(rng.integers(0, n)) if rng.random() < 0.5 else int(rng.integers(0, 64))
            b[at] ^= 1 << int(rng.integers(0, 8))
            cases.append(bytes(b))
        huge = bytearray(base)
        huge[11:15] = b"\xff\xff\xff\xff"       # a frame count no file could hold
        cases.append(bytes(huge))
    agree = 0
    for i, case in enumerate(cases):
        (tmp_path / "in.sela").write_bytes(case)
        p = subprocess.run([str(host_bin), "sela", str(tmp_path / "in.sela"), str(tmp_path / "out.sela")],
                           capture_output=True, text=True, timeout=60)
        try:
            info = codec.container_info(case)
            err = None
        except SelaB200Error as e:
            info, err = None, str(e)
        if p.returncode != 0:
            assert err is not None and p.stderr.strip() in err, (i, p.stderr, err)
        else:
            assert err is None, (i, err)
            back = (tmp_path / "out.sela").read_bytes()
            assert len(back) == info["n_bytes_used"] and back == case[:len(back)], (i, len(back), info)
        agree += 1
    assert agree == len(cases)
