"""More than one GPU behind the C ABI (selab200_init_devices) and behind NCCL (sela_b200.distributed's
device-resident scatter / gather): results must be byte-identical to one device's and to the reference's.
Skipped on a one-GPU box; run with  gpurun --gpus 2 -- python -m pytest tests/test_multi_device.py -q"""
import os
import socket

import numpy as np
import pytest

import oracle_lib as ol
import sela_b200
from sela_b200 import _lib, synth

pytestmark = pytest.mark.gpu
FRAME = 2048


def _n_gpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


needs2 = pytest.mark.skipif(_n_gpus() < 2, reason="needs two GPUs")


@pytest.fixture(scope="module")
def O():
    return ol.best()


def test_reinit_same_device_and_shutdown():
    """selab200_init is idempotent, survives a shutdown, and reports the device count."""
    L = _lib.lib()
    _lib.init(0)
    assert L.selab200_device_count() == 1
    L.selab200_shutdown()
    assert L.selab200_device_count() == 0
    _lib._initialised = None
    pcm = synth.sine_noise(44100, 2, n_frames=8, seed=5)
    d, w = sela_b200.encode_frames(pcm, 2)
    assert np.array_equal(sela_b200.decode_frames(d, w, 2), pcm.reshape(-1))


@needs2
def test_switching_the_device_rebuilds_the_context(O):
    """ADVICE r1: init(0) then init(1) must not keep device 0's streams and pools."""
    pcm = synth.sine_noise(44100, 2, n_frames=40, seed=6)
    d0, w0 = sela_b200.encode_frames(pcm, 2, device=0)
    d1, w1 = sela_b200.encode_frames(pcm, 2, device=1)
    assert d0.tobytes() == d1.tobytes() and np.array_equal(w0, w1)
    assert np.array_equal(sela_b200.decode_frames(d1, w1, 2, device=1), pcm.reshape(-1))
    assert np.array_equal(sela_b200.decode_frames(d0, w0, 2, device=0), pcm.reshape(-1))


@needs2
@pytest.mark.parametrize("channels,n_frames", [(2, 1531), (8, 613), (1, 700)])
def test_two_devices_equal_one_device_and_the_reference(O, channels, n_frames):
    pcm = synth.sine_noise(48000, channels, n_frames=n_frames, seed=9)
    if channels == 2:
        pcm[FRAME * 100:FRAME * 300, 1] = pcm[FRAME * 100:FRAME * 300, 0] - (pcm[FRAME * 100:FRAME * 300, 1] >> 6)
    d1, w1 = sela_b200.encode_frames(pcm, channels, device=0)
    d2, w2 = sela_b200.encode_frames(pcm, channels, device=[0, 1])
    assert _lib.lib().selab200_device_count() == 2
    assert d1.tobytes() == d2.tobytes() and np.array_equal(w1, w2)
    d_ref, w_ref = O.encode_frames(pcm, channels)
    assert d2.tobytes() == d_ref.tobytes() and np.array_equal(w2, w_ref)
    out2 = sela_b200.decode_frames(d2, w2, channels, device=[0, 1])
    assert np.array_equal(out2, O.decode_frames(d_ref, w_ref, channels))
    blob1 = sela_b200.encode_container(pcm, channels, 48000, device=0)
    blob2 = sela_b200.encode_container(pcm, channels, 48000, device=[1, 0])      # the other primary
    assert blob1.tobytes() == blob2.tobytes()
    info, out3 = sela_b200.decode_container(blob2, device=[1, 0])
    assert info["n_frames"] == n_frames and np.array_equal(out3, out2)
    with pytest.raises(_lib.SelaB200Error):                                      # capacity errors survive the device split
        sela_b200.encode_frames(pcm, channels, words_capacity=1000, device=[0, 1])
    _lib.init(0)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _nccl_worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    from sela_b200 import distributed as sd
    from sela_b200.device import DeviceCodec
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    channels, n_frames = 8, 1001
    pcm_dev = None
    if rank == 0:
        pcm = synth.sine_noise(48000, channels, n_frames=n_frames, seed=2)
        pcm_dev = torch.from_numpy(pcm.reshape(-1)).to(dev)
    (descs, words), t = sd.encode_sharded_device(pcm_dev, n_frames, channels, root=0)
    back, t2 = sd.decode_sharded_device(descs, words, n_frames, channels, root=0)
    if rank == 0:
        single = DeviceCodec(n_frames, channels, device=0)
        single.encode(pcm_dev)
        torch.cuda.synchronize()
        single.check_status()
        nw = int(single.words_used.item())
        same = bool(torch.equal(descs, single.descs)) and words.numel() == nw and bool(torch.equal(words, single.words[:nw]))
        out = torch.empty_like(pcm_dev)
        single.decode(out, nw)
        torch.cuda.synchronize()
        O = ol.best()
        d_ref, w_ref = O.encode_frames(pcm, channels)
        ref_same = descs.cpu().numpy().tobytes() == d_ref.tobytes() and np.array_equal(words.cpu().numpy().view(np.uint32), w_ref)
        q.put((same, bool(torch.equal(back, out)), ref_same))
    dist.barrier()
    dist.destroy_process_group()


@needs2
def test_nccl_scatter_encode_gather_equals_single_gpu_and_reference():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    try:
        res = q.get(timeout=240)
    finally:
        for p in procs:
            p.join(timeout=30)
            if p.is_alive():
                p.kill()
    for p in procs:
        assert p.exitcode == 0
    assert res == (True, True, True)


@needs2
def test_reference_main_on_two_devices_is_byte_identical(tmp_path):
    """The reference's own src/main.cpp, compiled against the mirror (bin/sela_refmain), with two GPUs behind the
    C ABI (SELAB200_DEVICES=0,1): `-e` and `-d` byte for byte against what the reference CLI wrote for the same
    WAV (digests in tests/golden/reference_cli.npz)."""
    import pathlib
    import subprocess
    from sela_b200 import wavio
    root = pathlib.Path(__file__).resolve().parent.parent
    refmain = root / "sela_b200" / "host" / "bin" / "sela_refmain"
    if not refmain.exists():
        pytest.skip("bin/sela_refmain not built (needs the reference tree at build time)")
    ref = ol.golden("reference_cli")
    wav = tmp_path / "oct.wav"
    wavio.write_wav(wav, synth.sine_noise(48000, 8, n_frames=700, seed=2), 48000)
    env = dict(os.environ, SELAB200_DEVICES="0,1")
    for cmd in ([refmain, "-e", wav, tmp_path / "a.sela"], [refmain, "-d", tmp_path / "a.sela", tmp_path / "a.wav"]):
        p = subprocess.run([str(c) for c in cmd], capture_output=True, text=True, timeout=600, env=env)
        assert p.returncode == 0, (cmd, p.stderr[-400:])
    for ext in ("sela", "wav"):
        got = np.frombuffer((tmp_path / ("a." + ext)).read_bytes(), np.uint8)
        assert ol.digest(got) == ref["oct700_" + ext], ext
