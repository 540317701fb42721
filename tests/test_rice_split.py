"""GPU parity of the second-generation Rice decoder (sela_b200/csrc/rice_vs.cuh): streams cut into S parts
by k_rice_split_index and decoded by k_rice_decode_vc, for every S, against the reference's decoder
(rice::RiceDecoder, src/rice/rice_decoder.cpp:11-52) -- including the streams it must hand back to the
general parser (periodic streams that never resynchronise, long unary runs, streams with more symbols per part than it keeps checkpoints for)."""
import numpy as np
import pytest

import oracle_lib as ol
import sela_b200
from sela_b200 import _lib, synth
from sela_b200.device import rice_decode_frames

pytestmark = pytest.mark.gpu
FRAME = 2048
SPLITS = ["0", "1", "2", "4", "8", "16"]


@pytest.fixture(scope="module")
def O():
    return ol.best()


def pack_stream(us, k):
    """rice_encoder.cpp:35-71 for a chosen k, vectorised: u >> k ones, a zero, k payload bits MSB first."""
    us = np.asarray(us, np.uint64)
    q = (us >> np.uint64(k)).astype(np.int64)
    lens = q + 1 + k
    starts = np.concatenate([[0], np.cumsum(lens)[:-1]])
    total = int(lens.sum())
    bits = np.zeros(total + (-total % 32), np.uint8)
    ones_idx = np.repeat(starts, q) + (np.arange(int(q.sum())) - np.repeat(np.cumsum(q) - q, q))
    bits[ones_idx] = 1
    for j in range(k):
        bits[starts + q + 1 + j] = ((us >> np.uint64(k - 1 - j)) & np.uint64(1)).astype(np.uint8)
    b = bits.reshape(-1, 32).astype(np.uint64)
    return (b << np.arange(32, dtype=np.uint64)).sum(axis=1).astype(np.uint32)


def zigzag(v):
    v = np.asarray(v, np.int64)
    return np.where(v >= 0, 2 * v, -2 * v - 1).astype(np.uint64)


def build_batch(streams, channels=1, gap_words=(0, 1, 2, 3, 5)):
    """streams: list of (k, words). Returns descriptors + arena with the streams at every 16-byte phase."""
    n = len(streams)
    assert n % channels == 0
    descs = np.zeros(n, _lib.DESC_DTYPE)
    arena = []
    at = 0
    for i, (k, w) in enumerate(streams):
        pad = gap_words[i % len(gap_words)]
        arena.append(np.full(pad, 0xFFFFFFFF, np.uint32))     # all-ones filler: must never be parsed
        at += pad
        d = descs[i]
        d["channel"] = i % channels
        d["parent_channel"] = i % channels
        d["lpc_order"] = 1
        d["refl_rice_param"] = 0
        d["refl_words"] = 1
        d["refl_offset"] = at
        arena.append(np.zeros(1, np.uint32))
        at += 1
        d["res_rice_param"] = k
        d["res_words"] = w.size
        d["samples"] = FRAME
        d["res_offset"] = at
        arena.append(w)
        at += w.size
    return descs, np.concatenate(arena)


def synthetic_streams(rng):
    out = []
    lap = lambda scale: np.round(rng.laplace(0, scale, FRAME)).astype(np.int64)
    # the BASELINE regime (k ~ 11) and its neighbours, chosen k around the optimum and away from it
    for scale, k in [(900, 10), (900, 11), (900, 12), (60, 5), (60, 7), (3, 1), (3, 2), (0.3, 0), (20000, 15), (20000, 13)]:
        out.append((k, zigzag(lap(scale))))
    # silence and constants: periodic streams in which a wrong-phase parse may never resynchronise
    out.append((0, zigzag(np.zeros(FRAME))))
    out.append((10, zigzag(np.full(FRAME, 1234))))
    out.append((3, zigzag(np.full(FRAME, -5))))
    out.append((6, zigzag(np.tile([37, -37], FRAME // 2))))
    out.append((11, zigzag(np.tile([1000, 1001, -999], FRAME // 3 + 1)[:FRAME])))
    # outliers: a few symbols longer than one 32-bit window, and very long runs
    v = lap(500); v[[5, 700, 701, 2047]] = [40000, -60000, 90000, -120000]; out.append((9, zigzag(v)))
    v = lap(30); v[::97] = 5000; out.append((4, zigzag(v)))
    v = lap(2); v[1000] = 3000; out.append((0, zigzag(v)))
    v = lap(800); v[256 * np.arange(1, 8)] = 70000; out.append((10, zigzag(v)))   # long symbols AT the part boundaries
    v = lap(800); v[256 * np.arange(1, 8) - 1] = -70000; out.append((10, zigzag(v)))
    # loud then quiet: parts with very different bit densities
    v = np.concatenate([lap(8000)[:300], lap(3)[:FRAME - 300]]); out.append((4, zigzag(v)))
    v = np.concatenate([lap(2)[:1800], lap(6000)[:248]]); out.append((3, zigzag(v)))
    # k extremes
    out.append((19, zigzag(rng.integers(-(1 << 19), 1 << 19, FRAME))))
    out.append((24, zigzag(rng.integers(-(1 << 23), 1 << 23, FRAME))))
    out.append((31, rng.integers(0, 1 << 31, FRAME).astype(np.uint64)))
    # full-scale noise: the longest streams 16-bit audio produces
    out.append((16, zigzag(rng.integers(-65535, 65536, FRAME))))
    return [(k, pack_stream(us, k), us) for k, us in out]


@pytest.mark.parametrize("split", SPLITS)
def test_split_decoder_synthetic_streams(O, monkeypatch, split):
    monkeypatch.setenv("SELAB200_RICE_SPLIT", split)
    rng = np.random.default_rng(11)
    streams = synthetic_streams(rng) * 3                      # > one warp of streams at every S
    descs, arena = build_batch([(k, w) for k, w, _ in streams])
    res, flagged = rice_decode_frames(descs, arena, 1)
    for i, (k, w, us) in enumerate(streams):
        want = O.rice_decode(w, k, FRAME)
        assert np.array_equal(res[i], want), (split, i, k)
    u = np.asarray(streams[0][2], np.uint64)
    assert np.array_equal(res[0], ((u >> np.uint64(1)).astype(np.int64) ^ -(u & np.uint64(1)).astype(np.int64)).astype(np.int32))
    if split not in ("0",):
        assert flagged < len(streams)                          # the fast decoder did most of the work


@pytest.mark.parametrize("split", SPLITS)
def test_split_decoder_encoded_batch(O, monkeypatch, split):
    """Streams produced by the encoder (stereo, difference coding, all order classes)."""
    monkeypatch.setenv("SELAB200_RICE_SPLIT", split)
    pcm = synth.sine_noise(44100, 2, n_frames=150, seed=3)
    pcm[FRAME * 20:FRAME * 40] //= 64                          # a quiet passage: small k
    pcm[FRAME * 60:FRAME * 70] = 0                             # silence: k = 0, 64-word streams
    pcm[FRAME * 80:FRAME * 90, 1] = pcm[FRAME * 80:FRAME * 90, 0] + 3   # difference-coded frames
    d, w = O.encode_frames(pcm, 2)
    res, flagged = rice_decode_frames(d, w, 2)
    for i in range(0, d.size, 7):
        want = O.rice_decode(w[int(d[i]["res_offset"]):int(d[i]["res_offset"]) + int(d[i]["res_words"])],
                             int(d[i]["res_rice_param"]), FRAME)
        assert np.array_equal(res[i], want), (split, i)
    out = sela_b200.decode_frames(d, w, 2)                     # and the whole decode chain on top of it
    assert np.array_equal(out, O.decode_frames(d, w, 2))
    if split not in ("0",):
        assert flagged <= d.size // 4, flagged


def test_split_decoder_truncated_stream_is_rejected(O, monkeypatch):
    for split in ("1", "8"):
        monkeypatch.setenv("SELAB200_RICE_SPLIT", split)
        rng = np.random.default_rng(4)
        us = zigzag(np.round(rng.laplace(0, 900, FRAME)).astype(np.int64))
        w = pack_stream(us, 11)
        descs, arena = build_batch([(11, w[:w.size // 2])] * 4)
        with pytest.raises(_lib.SelaB200Error) as e:
            rice_decode_frames(descs, arena, 1)
        assert e.value.status == -6
