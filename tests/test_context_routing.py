"""Which device and context each C ABI call runs on.

The *_device forms run on the device that owns the caller's buffers, which need not be the primary. The
host-buffer and container calls split their frames over every initialised device, each device pipelining
its block in chunks. Their results and their errors must not depend on either. Container handles belong
to the primary device, whichever thread closes them. All but the last test need two GPUs."""
import ctypes as C
import threading

import numpy as np
import pytest

import sela_b200
from sela_b200 import _lib, codec, synth
from sela_b200._lib import FRAME, INFO_DTYPE, SelaB200Error

pytestmark = pytest.mark.gpu


def _n_gpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


needs2 = pytest.mark.skipif(_n_gpus() < 2, reason="needs two GPUs")


def _pcm(channels, n_frames, seed):
    pcm = synth.sine_noise(48000, channels, n_frames=n_frames, seed=seed)
    if channels == 2:                                     # some frames where the difference channel wins
        pcm[FRAME * 40:FRAME * 90, 1] = pcm[FRAME * 40:FRAME * 90, 0] - (pcm[FRAME * 40:FRAME * 90, 1] >> 6)
    return pcm


def _device_calls(dev, pcm, channels):
    """Every *_device call on buffers of cuda:`dev`, through the C ABI as the library is initialised now."""
    import torch
    L = _lib.lib()
    d = torch.device("cuda", dev)
    n_frames = pcm.shape[0] // FRAME
    n_sub = n_frames * channels
    cap = L.selab200_encode_words_bound(n_frames, channels)
    d_pcm = torch.from_numpy(pcm.reshape(-1)).to(d)
    descs = torch.zeros(n_sub * 32, dtype=torch.uint8, device=d)
    words = torch.zeros(cap + 8, dtype=torch.int32, device=d)
    used = torch.zeros(1, dtype=torch.int64, device=d)
    status = torch.zeros(3, dtype=torch.int32, device=d)
    enc_ws_bytes = L.selab200_encode_workspace_bytes(n_frames, channels)
    dec_ws_bytes = L.selab200_decode_workspace_bytes(n_frames, channels)
    enc_ws = torch.zeros(enc_ws_bytes, dtype=torch.uint8, device=d)
    dec_ws = torch.zeros(dec_ws_bytes, dtype=torch.uint8, device=d)
    out = torch.zeros_like(d_pcm)
    residues = torch.zeros(n_sub * FRAME, dtype=torch.int32, device=d)
    stream = C.c_void_p(torch.cuda.current_stream(d).cuda_stream)
    _lib.check(L.selab200_encode_frames_device(d_pcm.data_ptr(), n_frames, channels, descs.data_ptr(),
                                               words.data_ptr(), cap, used.data_ptr(), status.data_ptr(),
                                               enc_ws.data_ptr(), enc_ws_bytes, stream))
    torch.cuda.synchronize(d)
    nw = int(used.item())
    _lib.check(L.selab200_decode_frames_device(descs.data_ptr(), n_frames, channels, words.data_ptr(), nw,
                                               out.data_ptr(), status.data_ptr() + 4, dec_ws.data_ptr(),
                                               dec_ws_bytes, stream))
    _lib.check(L.selab200_rice_decode_frames_device(descs.data_ptr(), n_frames, channels, words.data_ptr(), nw,
                                                    residues.data_ptr(), status.data_ptr() + 8, stream))
    torch.cuda.synchronize(d)
    flagged = C.c_uint32(0)
    _lib.check(L.selab200_rice_decode_flagged(C.addressof(flagged)))
    assert status.cpu().tolist() == [0, 0, 0]
    return (descs.cpu().numpy().tobytes(), words[:nw].cpu().numpy().tobytes(), out.cpu().numpy().tobytes(),
            residues.cpu().numpy().tobytes(), flagged.value)


@needs2
@pytest.mark.parametrize("channels", [2, 3])
def test_device_forms_on_a_secondary_device_equal_the_primary(channels):
    pcm = _pcm(channels, 37, 4)
    _lib.init([0, 1])
    try:
        on1 = _device_calls(1, pcm, channels)
        on0 = _device_calls(0, pcm, channels)
    finally:
        _lib.init(0)
    assert on1 == on0
    assert np.frombuffer(on0[2], np.int16).tobytes() == pcm.reshape(-1).tobytes()


@needs2
@pytest.mark.parametrize("channels,n_frames", [(2, 530), (3, 517)])
def test_many_chunks_on_two_devices_equal_one_device(monkeypatch, channels, n_frames):
    """SELAB200_CHUNK_FRAMES makes every device run many chunks; blocks of at least 256 frames per device are
    what sends the host-buffer calls to all devices."""
    pcm = _pcm(channels, n_frames, 11)
    monkeypatch.setenv("SELAB200_CHUNK_FRAMES", "16")
    try:
        d1, w1 = sela_b200.encode_frames(pcm, channels, device=0)
        out1 = sela_b200.decode_frames(d1, w1, channels, device=0)
        blob1 = sela_b200.encode_container(pcm, channels, 48000, device=0)
        out3 = sela_b200.decode_container(blob1, device=0)[1]
        d2, w2 = sela_b200.encode_frames(pcm, channels, device=[0, 1])
        out2 = sela_b200.decode_frames(d1, w1, channels, device=[0, 1])
        blob2 = sela_b200.encode_container(pcm, channels, 48000, device=[0, 1])
        out4 = sela_b200.decode_container(blob1, device=[0, 1])[1]
    finally:
        _lib.init(0)
    assert d1.tobytes() == d2.tobytes() and np.array_equal(w1, w2)
    assert np.array_equal(out1, pcm.reshape(-1)) and np.array_equal(out2, out1)
    assert blob1.tobytes() == blob2.tobytes()
    assert np.array_equal(out3, out1) and np.array_equal(out4, out1)


def _error(fn):
    with pytest.raises(SelaB200Error) as e:
        fn()
    return e.value.status, str(e.value)


@needs2
def test_errors_on_two_devices_equal_one_device():
    channels, n_frames = 2, 600
    pcm = _pcm(channels, n_frames, 13)
    blob = sela_b200.encode_container(pcm, channels, 48000, device=0)
    _, offsets = codec.container_frame_offsets(blob)
    bad = blob.copy()
    bad[int(offsets[n_frames * 3 // 4]) + 4 + 6] = 200     # lpc_order of a subframe in the second device's block
    errors = {}
    try:
        for devices in ([0], [0, 1]):
            errors[len(devices)] = (
                _error(lambda: sela_b200.decode_container(bad, device=devices)),
                _error(lambda: sela_b200.encode_frames(pcm, channels, words_capacity=1000, device=devices)),
                _error(lambda: sela_b200.encode_container(pcm, channels, 48000, capacity=blob.size // 2,
                                                          device=devices)),
            )
    finally:
        _lib.init(0)
    assert errors[1] == errors[2]
    assert [s for s, _ in errors[1]] == [-6, -4, -4]      # BITSTREAM, CAPACITY, CAPACITY


def test_container_closed_on_another_thread_is_reused():
    """selab200_container_close from a thread that never selected a device returns the handle's buffers to the
    primary's spare list; the next open takes them and decodes correctly."""
    L = _lib.lib()
    _lib.init(0)
    pcms = [_pcm(2, 9, 21), _pcm(2, 5, 22)]
    blobs = [sela_b200.encode_container(p, 2, 48000) for p in pcms]
    for pcm, blob in zip(pcms, blobs):
        info = np.zeros(1, INFO_DTYPE)
        handle = C.c_void_p(0)
        _lib.check(L.selab200_container_open(blob.ctypes.data, blob.size, C.addressof(handle), info.ctypes.data))
        out = np.empty(pcm.size, np.int16)
        _lib.check(L.selab200_container_decode(handle, out.ctypes.data))
        t = threading.Thread(target=L.selab200_container_close, args=(handle,))
        t.start()
        t.join()
        assert np.array_equal(out, pcm.reshape(-1))
    assert np.array_equal(sela_b200.decode_container(blobs[0])[1], pcms[0].reshape(-1))
