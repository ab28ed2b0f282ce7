"""Device ingest (SURVEY.md 8f rank 3): soundml-io's layout pass and the fused
decode-block -> resample loop on the GPU, against the oracle.  The layout pass is
copy / one rounded multiply: bit-exact.  The fused loop is held to the resampler's
bar (1e-5 of peak) and to the reference's chunking law (a chunked read equals the
whole read)."""
import numpy as np
import pytest

from golden_util import peak_rel_err
from oracle import io_oracle, resample_oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sb(lib):
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return lib


def _block(frames, channels, dtype, seed=3):
    rng = np.random.default_rng(seed)
    return rng.uniform(-1, 1, (frames, channels)).astype(dtype)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("channels", [1, 2, 3, 6])
@pytest.mark.parametrize("mode", ["planar", "mono"])
def test_layout_is_bit_exact(sb, dtype, channels, mode):
    import torch
    for frames in (1, 7, 4096, 10001):
        b = _block(frames, channels, dtype)
        ref = io_oracle.layout(b, mode)
        got = sb.Io.layout(b, mode)                       # host block -> device planar
        assert got.is_cuda and tuple(got.shape) == ref.shape
        assert np.array_equal(got.cpu().numpy(), ref)
        got_h = sb.Io.layout(b, mode, device="host")      # host -> host
        assert isinstance(got_h, np.ndarray) and np.array_equal(got_h, ref)
        got_d = sb.Io.layout(torch.from_numpy(b).cuda(), mode)   # device -> device
        assert np.array_equal(got_d.cpu().numpy(), ref)


def test_layout_staging_is_per_device(sb):
    """The layout call keeps its staging per thread and per device: after a large block on
    device 0, a smaller one on device 1 must not reuse device 0's buffer."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    for device, frames in ((0, 50000), (1, 3000)):
        b = _block(frames, 2, np.float32, device)
        ref = io_oracle.layout(b, "planar")
        with torch.cuda.device(device):
            got = sb.Io.layout(b, "planar", device=f"cuda:{device}")                      # host -> device
            assert got.device.index == device and np.array_equal(got.cpu().numpy(), ref)
            got_h = sb.Io.layout(torch.from_numpy(b).to(f"cuda:{device}"), "planar", device="host")
            assert np.array_equal(got_h, ref)                                             # device -> host


def test_layout_into_a_longer_destination(sb):
    import torch
    b0, b1 = _block(1000, 2, np.float32, 1), _block(500, 2, np.float32, 2)
    out = torch.zeros((2, 1500), dtype=torch.float32, device="cuda")
    sb.Io.layout(b0, "planar", out=out, out_off=0)
    sb.Io.layout(b1, "planar", out=out, out_off=1000)
    assert np.array_equal(out.cpu().numpy(), np.concatenate([b0, b1]).T)
    with pytest.raises(ValueError):
        sb.Io.layout(b1, "planar", out=out, out_off=1200)


def test_block_sizing_matches_the_reference_rule(sb):
    for channels, elt, adv in [(1, 4, 0), (2, 4, 0), (2, 8, 0), (6, 4, 0), (1, 4, 100), (2, 4, 50000),
                               (1, 4, 5_000_000), (64, 8, 0)]:
        assert sb.Io.decode_block_frames(channels, elt, adv) == io_oracle.decode_block_frames(channels, elt, adv)
    assert sb.Io.decode_block_frames(2, 4) == 524288          # 4 MB of stereo float32
    assert sb.Io.decode_block_frames(1, 4) == 1048576         # capped at 1 Mi frames


@pytest.mark.parametrize("rates,mode", [((44100, 16000), "mono"), ((44100, 22050), "planar"),
                                        ((48000, 8000), "planar"), ((22050, 22050), "mono")])
def test_fused_ingest_equals_offline_resample(sb, rates, mode):
    """decode_step law: blocks fed one by one == layout of the whole signal, then
    Resample.apply; and the oracle's float64 evaluation within 1e-5 of peak."""
    sr, target = rates
    frames, channels = 60000, 2
    t = np.arange(frames)
    sig = np.stack([0.5 * np.sin(2 * np.pi * 440 * t / sr), 0.3 * np.sin(2 * np.pi * 1000 * t / sr)], 1)
    sig = (sig + 0.05 * _block(frames, channels, np.float64, 9)).astype(np.float32)
    whole = io_oracle.layout(sig, mode)
    for block in (4096, 17000, 60000):
        rd = sb.Io.Ingest(channels=channels, sample_rate=sr, target=target, mode=mode, max_block=block)
        got = rd.read(sig[i:i + block] for i in range(0, frames, block)).cpu().numpy()
        if sr == target:
            assert np.array_equal(got, whole)
            continue
        cfg = sb.Resample.Config.create(sample_rate=sr, target=target)
        off = sb.Resample.apply(cfg, whole)
        assert got.shape == off.shape == (whole.shape[0], -(-frames * cfg.l // cfg.m))
        assert peak_rel_err(got, off) <= 1e-5, (rates, block)
    if sr != target:
        from test_resample_oracle import oracle_stages
        cfg = sb.Resample.Config.create(sample_rate=sr, target=target)
        ref = resample_oracle.apply_plan(whole.astype(np.float64), oracle_stages(cfg), cfg.l, cfg.m)
        assert peak_rel_err(got, ref) <= 1e-5


def test_ingest_argument_checks(sb):
    rd = sb.Io.Ingest(channels=2, sample_rate=44100, target=22050, max_block=1000)
    with pytest.raises(ValueError):
        rd.feed(np.zeros((10, 3), np.float32))
    with pytest.raises(ValueError):
        rd.feed(np.zeros((1001, 2), np.float32))
    assert rd.feed(np.zeros((0, 2), np.float32)) is None
    rd.finish()
    with pytest.raises(ValueError):
        rd.feed(np.zeros((10, 2), np.float32))


def test_reader_decodes_into_pinned_staging_blocks(sb):
    """The decode loop as soundml-io runs it (soundml_io.ml:742-807): the decoder writes block
    i + 1 into the other pinned staging block while block i is uploaded and resampled; nothing
    but ``submit`` touches the data.  The pieces concatenate to the offline result."""
    import torch
    sr, target, channels, frames = 44100, 16000, 2, 150000
    rng = np.random.default_rng(3)
    sig = rng.uniform(-1, 1, (frames, channels)).astype(np.float32)
    rd = sb.Io.Ingest(channels=channels, sample_rate=sr, target=target, mode="mono", max_block=8192)
    assert rd.max_block == 8192
    pieces, blocks = [], []
    for i in range(0, frames, 8192):
        blk = rd.staging()
        blocks.append(blk.ctypes.data)
        n = min(8192, frames - i)
        blk[:n] = sig[i:i + n]                                 # "sf_readf_float" into pinned memory
        p = rd.submit(n)
        if p is not None:
            pieces.append(p)
    assert len(set(blocks)) == 2 and blocks[0] != blocks[1] and blocks[0] == blocks[2]   # two blocks, alternating
    tail = rd.finish()
    if tail is not None:
        pieces.append(tail)
    got = torch.cat(pieces, dim=-1).cpu().numpy()
    cfg = sb.Resample.Config.create(sample_rate=sr, target=target)
    off = sb.Resample.apply(cfg, io_oracle.layout(sig, "mono"))
    assert got.shape == off.shape == (1, -(-frames * cfg.l // cfg.m))
    assert peak_rel_err(got, off) <= 1e-5
    with pytest.raises(ValueError):
        rd.submit(10)
    # native rate, float64, planar: the layout pass alone, bit for bit
    rd = sb.Io.Ingest(channels=3, sample_rate=48000, target=None, max_block=5000, dtype=np.float64)
    sig64 = rng.uniform(-1, 1, (12345, 3))
    got = rd.read(sig64[i:i + 5000] for i in range(0, 12345, 5000)).cpu().numpy()
    assert np.array_equal(got, io_oracle.layout(sig64, "planar"))
