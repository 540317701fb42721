"""Pins the plain-C oracle (oracle/sela_oracle.c) against what the UNMODIFIED reference computed on the
same inputs (stored in tests/golden/reference_stages.npz by tests/golden/make_golden.py), and against
SURVEY.md 8a's KAT table.  CPU only."""
import numpy as np
import pytest

import oracle_lib as ol
import signals
from sela_b200 import synth

# SURVEY.md 8(a) known answers: (order, refl k, refl words, res k, res words, res word0, res last, refl fnv, res fnv)
KAT = {
    "sine_deg": (17, 4, 3, 7, 552, 0xFF6EFF00, 0x00000010, 0x0BC50C3B, 0xFAF0DFE3),
    "zeros": (1, 0, 1, 0, 64, 0, 0, 0x4B95F515, 0xE6A1D1C5),
    "dc_1234": (1, 6, 1, 10, 832, 0xCC9664B3, 0x25992CC9, 0x1DAF5698, 0xFF0C5DC5),
    "cosine_deg": (16, 4, 3, 7, 585, 0xFFFFFFFF, 0x00000019, 0x4F1CBBE0, 0x10A3227D),
    "impulse0": (1, 5, 1, 4, 448, 0xFFFFFFFF, 0x00000000, 0xBD7CAAD0, 0x266C2942),
}


# ---- the inputs (make_golden.py runs the reference on exactly these) ----
def dc_levels():
    return list(range(-32768, 32768, 257)) + [-32768, -1, 1, 32767]


def rice_inputs():
    rng = np.random.default_rng(5)
    out = [rng.integers(-scale, scale + 1, n).astype(np.int32)
           for n, scale in [(100, 400), (1, 5), (2048, 3), (2048, 70000), (333, 1 << 20), (17, 0)]]
    # the reference's own test input shape: 100 values in [200, 400] (test/ricetests.cpp:11-13)
    out.append((200 + rng.integers(0, 201, 100)).astype(np.int32))
    return out


def batch_pcm(channels):
    pcm = synth.sine_noise(44100, channels, n_frames=12, seed=3)
    if channels == 2:                       # make some frames favour difference coding
        pcm[2048 * 3:2048 * 6, 1] = pcm[2048 * 3:2048 * 6, 0] - (pcm[2048 * 3:2048 * 6, 1] >> 6)
        pcm[2048 * 6:2048 * 7, 1] = pcm[2048 * 6:2048 * 7, 0]
    return pcm


def _code(O, s):
    a = O.lpc_analyse(s)
    kq, wq = O.rice_encode(a["q"])
    kr, wr = O.rice_encode(a["res"])
    return a, kq, wq, kr, wr


@pytest.mark.parametrize("name", sorted(KAT))
@pytest.mark.parametrize("which", ["port", "ref"])
def test_kat_table(name, which):
    if which == "port":
        a, kq, wq, kr, wr = _code(ol.load("port"), signals.families()[name])
        order = a["order"]
    else:
        ref = ol.golden("reference_stages")
        g = lambda f: ref["fam_%s_%s" % (name, f)]
        order, kq, wq, kr, wr = int(g("order")), int(g("kq")), g("wq"), int(g("kr")), g("wr")
    got = (order, kq, len(wq), kr, len(wr), int(wr[0]), int(wr[-1]), ol.fnv1a32(wq), ol.fnv1a32(wr))
    assert got == KAT[name]


def test_families_port_equals_reference():
    P, ref = ol.load("port"), ol.golden("reference_stages")
    for name, s in signals.families().items():
        g = lambda f: ref["fam_%s_%s" % (name, f)]
        a = P.lpc_analyse(s)
        assert a["order"] == int(g("order")), name
        assert np.array_equal(a["q"], g("q")), name
        assert np.array_equal(a["c"], g("c")), name
        assert np.array_equal(a["res"], g("res")), name
        for x, part in ((a["q"], "q"), (a["res"], "r")):
            k1, w1 = P.rice_encode(x)
            assert k1 == int(g("k" + part)) and np.array_equal(w1, g("w" + part)), name
            assert np.array_equal(P.rice_decode(w1, k1, x.size), x), name
            assert ol.digest(x) == g("decoded_" + part), name       # the reference decoded its stream to x
        assert np.array_equal(P.lpc_synthesise(a["res"], a["order"], a["q"]), s), name
        assert ol.digest(s) == g("synthesised"), name


def test_random_subframes_port_equals_reference():
    P, ref = ol.load("port"), ol.golden("reference_stages")
    for i, s in enumerate(signals.random_frames(300, seed=11)):
        a = P.lpc_analyse(s)
        assert a["order"] == ref["rand_order"][i], i
        assert np.array_equal(a["q"], ref["rand_q"][i, :a["order"]]) and not ref["rand_q"][i, a["order"]:].any(), i
        assert ol.digest(a["res"]) == ref["rand_res"][i], i


def test_dc_levels_port_equals_reference():
    """Constant frames: x-mean is pure rounding noise, the case where summation order
    changes q[0] (SURVEY.md 7.3-H1)."""
    P, ref = ol.load("port"), ol.golden("reference_stages")
    levels = dc_levels()
    assert list(ref["dc_level"]) == levels
    for i, level in enumerate(levels):
        a = P.lpc_analyse(np.full(2048, level, np.int32))
        assert (a["order"], list(a["q"])) == (ref["dc_order"][i], list(ref["dc_q"][i, :ref["dc_order"][i]])), level
        assert ol.digest(a["res"]) == ref["dc_res"][i], level


def test_rice_port_equals_reference_random():
    P, ref = ol.load("port"), ol.golden("reference_stages")
    for i, x in enumerate(rice_inputs()):
        k1, w1 = P.rice_encode(x)
        assert k1 == ref["rice_%d_k" % i] and np.array_equal(w1, ref["rice_%d_words" % i]), i
        assert np.array_equal(P.rice_decode(w1, k1, x.size), x), i
        assert ol.digest(x) == ref["rice_%d_decoded" % i], i


@pytest.mark.parametrize("channels", [1, 2, 3, 8])
def test_batch_port_equals_reference(channels):
    P, ref = ol.load("port"), ol.golden("reference_stages")
    pcm = batch_pcm(channels)
    d1, w1 = P.encode_frames(pcm, channels, threads=3)
    assert d1.tobytes() == ref["batch%d_descs" % channels].tobytes()
    assert ol.digest(w1) == ref["batch%d_words" % channels]
    if channels == 2:
        assert set(d1["subframe_type"]) == {0, 1}
    assert np.array_equal(P.decode_frames(d1, w1, channels), pcm.reshape(-1))
    assert ol.digest(pcm.reshape(-1)) == ref["batch%d_decoded" % channels]


def test_frame_roundtrip_reference_test_shape():
    """test/frametests.cpp:8-38: both channels the same sine -> the difference channel is
    all-zero (NaN path, order 1) and wins."""
    P = ol.load("port")
    s = synth.config1_frame()
    descs, words = P.frame_encode_i32([s, s])
    assert list(descs["subframe_type"]) == [0, 1] and list(descs["parent_channel"]) == [0, 0]
    assert descs["lpc_order"][1] == 1 and descs["res_words"][1] == 64
    out = P.frame_decode_i32(descs, words)
    assert np.array_equal(out[0], s) and np.array_equal(out[1], s)


def test_port_roundtrip_families():
    P = ol.load("port")
    for name, s in signals.families().items():
        a = P.lpc_analyse(s)
        assert np.array_equal(P.lpc_synthesise(a["res"], a["order"], a["q"]), s), name
        k, w = P.rice_encode(a["res"])
        assert np.array_equal(P.rice_decode(w, k, s.size), a["res"]), name
