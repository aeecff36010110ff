"""GPU: the peak decode (csrc/peaks.cu) bit for bit against the numpy reference of tests/peaks_ref.py, its C ABI error paths, and the
serving calls built on it (KeypointsGauss.peaks, Prediction.peaks)."""
import ctypes as C
import warnings

import numpy as np
import pytest
import torch

import hulk_keypoints_b200 as hk
from hulk_keypoints_b200 import _lib, ops
from hulk_keypoints_b200.prediction import Prediction
from peaks_ref import peak_decode_ref, peak_mask

warnings.filterwarnings("ignore")
pytestmark = pytest.mark.gpu

RS = [1, 2, 4, 8, 16]
NS = [1, 7, 64, 256]
SHAPES = [(64, 4, 480, 640), (16, 32, 960, 1280), (2, 3, 33, 47), (1, 1, 1, 1), (1, 1, 1, 700)]


def _maps_checked(M):
    """All maps of a small batch; for the large shapes a fixed spread of maps (the kernels treat every map alike and independently)."""
    return np.arange(M) if M <= 64 else np.unique(np.linspace(0, M - 1, 12).astype(np.int64))


def assert_matches(heat, N, thr, r, maps=None, got=None):
    B, K, H, W = heat.shape
    yx, score, count = got if got is not None else ops.peak_decode(heat, N, thr, r)
    sel = np.arange(B * K) if maps is None else maps
    h = heat.reshape(B * K, H, W)[torch.as_tensor(sel, device=heat.device)].cpu().numpy()
    ryx, rscore, rcount = peak_decode_ref(h, N, thr, r)
    gyx = yx.reshape(B * K, N, 2).cpu().numpy()[sel]
    gscore = score.reshape(B * K, N).cpu().numpy()[sel]
    gcount = count.reshape(B * K).cpu().numpy()[sel]
    assert np.array_equal(gcount, rcount), (np.flatnonzero(gcount != rcount)[:5], gcount[:8], rcount[:8])
    assert np.array_equal(gyx, ryx), np.argwhere(gyx != ryx)[:5]
    assert np.array_equal(gscore, rscore)
    return rcount


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_shapes_uniform_random_all_r_and_n(shape):
    B, K, H, W = shape
    heat = torch.rand(shape, device="cuda", generator=_gen(1))
    sel = _maps_checked(B * K)
    h = heat.reshape(B * K, H, W)[torch.as_tensor(sel, device="cuda")].cpu().numpy()
    for r in RS:
        mask = peak_mask(h, r, 0.5)
        ref = peak_decode_ref(h, max(NS), 0.5, r, mask=mask)
        for N in NS:
            yx, score, count = ops.peak_decode(heat, N, 0.5, r)
            assert np.array_equal(count.reshape(-1).cpu().numpy()[sel], np.minimum(ref[2], N)), (r, N)
            assert np.array_equal(yx.reshape(B * K, N, 2).cpu().numpy()[sel], ref[0][:, :N]), (r, N)
            assert np.array_equal(score.reshape(B * K, N).cpu().numpy()[sel], ref[1][:, :N]), (r, N)
            if H * W >= 4096 and N < 256 and r == 1:
                assert (count.reshape(-1)[torch.as_tensor(sel, device="cuda")] == N).all()   # more candidates than N in a tile


@pytest.mark.parametrize("r", RS)
def test_quantised_plateaus(r):
    heat = torch.randint(0, 4, (2, 3, 100, 300), device="cuda", generator=_gen(2)).float() / 3
    for N in (7, 256):
        assert_matches(heat, N, 1 / 3, r)


def test_constant_map_has_one_peak_at_origin():
    heat = torch.full((2, 2, 70, 260), 0.75, device="cuda")
    for r in RS:
        yx, score, count = ops.peak_decode(heat, 4, 0.5, r)
        assert (count == 1).all()
        assert (yx[..., 0, :] == 0).all() and (score[..., 0] == 0.75).all()
        assert (yx[..., 1:, :] == -1).all() and torch.isinf(score[..., 1:]).all() and (score[..., 1:] < 0).all()


@pytest.mark.parametrize("r", RS)
def test_nan_and_infinities(r):
    g = _gen(3)
    heat = torch.rand((2, 2, 90, 200), device="cuda", generator=g)
    u = torch.rand(heat.shape, device="cuda", generator=g)
    heat[u < 0.03] = float("nan")
    heat[(u >= 0.03) & (u < 0.05)] = float("inf")
    heat[(u >= 0.05) & (u < 0.08)] = -float("inf")
    for N in (7, 256):
        assert_matches(heat, N, 0.25, r)
    assert_matches(torch.full((1, 1, 40, 140), float("nan"), device="cuda"), 7, 0.0, r)   # nothing is a peak


@pytest.mark.parametrize("r", RS)
def test_planted_peaks_on_tile_edges_borders_and_corners(r):
    B, K, H, W = 1, 2, 100, 300   # tiles of 32 x 128: edges at rows 31|32, 63|64, 95|96 and columns 127|128, 255|256
    heat = torch.rand((B, K, H, W), device="cuda", generator=_gen(4)) * 0.1
    spots = [(0, 0), (0, W - 1), (H - 1, 0), (H - 1, W - 1), (31, 127), (32, 128), (63, 255), (64, 256), (95, 40), (96, 41),
             (0, 128), (50, 0), (50, W - 1), (H - 1, 127), (31, 200), (32, 200)]
    for i, (y, x) in enumerate(spots):
        heat[:, :, y, x] = 0.5 + 0.01 * i
    heat[:, 1, 32, 129] = 0.5 + 0.01 * 5   # an equal value right after a planted peak: the earlier one wins
    for N in (1, 7, 64):
        assert_matches(heat, N, 0.3, r)


@pytest.mark.parametrize("r", [1, 4, 8, 16])
def test_realistic_gaussian_blobs(r):
    B, K, H, W, blobs = 4, 4, 480, 640, 6
    g = torch.Generator().manual_seed(5)
    uv = torch.stack([torch.rand(B * blobs, K, generator=g) * (W - 1), torch.rand(B * blobs, K, generator=g) * (H - 1)], -1).cuda()
    t = ops.gauss_targets(uv, H, W, 8.0, out_dtype=torch.float32)            # (B*blobs, K, H, W)
    heat = t.view(B, blobs, K, H, W).amax(1).contiguous()
    for N in (1, 7, 64):
        rc = assert_matches(heat, N, 0.5, r)
        if N == 64:
            assert rc.min() >= 1 and rc.max() > 1   # several instances per channel are found


@pytest.mark.parametrize("r", RS)
def test_top1_equals_argmax_decode(r):
    g = _gen(6)
    for heat in (torch.rand((3, 4, 97, 333), device="cuda", generator=g),
                 torch.randint(0, 5, (3, 4, 97, 333), device="cuda", generator=g).float() / 4,
                 torch.rand((2, 2, 480, 640), device="cuda", generator=g)):
        yx, score, count = ops.peak_decode(heat, 1, -1.0, r)
        ayx, amax = ops.argmax_decode(heat, want_max=True)
        assert (count == 1).all()
        assert torch.equal(yx[..., 0, :], ayx) and torch.equal(score[..., 0], amax)


def test_two_calls_identical_bytes():
    heat = torch.rand((8, 4, 480, 640), device="cuda", generator=_gen(7))
    for r, N in ((1, 256), (4, 64), (16, 7)):
        a = [t.clone() for t in ops.peak_decode(heat, N, 0.5, r)]
        b = ops.peak_decode(heat, N, 0.5, r)
        torch.cuda.synchronize()
        assert all(torch.equal(x.view(torch.uint8), y.view(torch.uint8)) for x, y in zip(a, b))


def test_c_abi_error_paths():
    lib = _lib.lib()
    heat = torch.rand((1, 2, 40, 50), device="cuda")
    yx = torch.empty((1, 2, 8, 2), device="cuda", dtype=torch.int32)
    score = torch.empty((1, 2, 8), device="cuda")
    count = torch.empty((1, 2), device="cuda", dtype=torch.int32)
    nbytes = int(lib.hk_peak_workspace_bytes(1, 2, 40, 50, 8, 3))
    ws = torch.empty(nbytes, device="cuda", dtype=torch.uint8)
    s = _lib.stream_ptr()
    p = _lib.ptr

    def call(*a):
        return lib.hk_peak_decode(*a)

    ok = (p(heat), 1, 2, 40, 50, 8, 3, C.c_float(0.5), p(yx), p(score), p(count), p(ws), nbytes, s)
    assert call(*ok) == 0
    bad = [
        (p(heat), 0, 2, 40, 50, 8, 3, C.c_float(0.5), p(yx), p(score), p(count), p(ws), nbytes, s),           # bad shape
        (p(heat), 1, 2, 40, 50, 8, 3, C.c_float(0.5), p(yx), p(score), p(count), p(ws), nbytes - 1, s),       # workspace too small
        (None, 1, 2, 40, 50, 8, 3, C.c_float(0.5), p(yx), p(score), p(count), p(ws), nbytes, s),               # null heat
        (p(heat), 1, 2, 40, 50, 8, 3, C.c_float(0.5), p(yx), None, p(count), p(ws), nbytes, s),                # null score
        (p(heat), 1, 2, 40, 50, 8, 3, C.c_float(0.5), p(yx), p(score), p(count), None, nbytes, s),             # null workspace
        (p(heat), 1, 2, 40, 50, 0, 3, C.c_float(0.5), p(yx), p(score), p(count), p(ws), nbytes, s),            # N = 0
        (p(heat), 1, 2, 40, 50, 8, 17, C.c_float(0.5), p(yx), p(score), p(count), p(ws), nbytes, s),           # r = 17
        (p(heat), 1, 2, 40, 50, 8, 3, C.c_float(float("nan")), p(yx), p(score), p(count), p(ws), nbytes, s),   # NaN threshold
    ]
    for args in bad:
        assert call(*args) < 0
        assert lib.hk_last_error().decode().startswith("hk_peak_decode")
    torch.cuda.synchronize()


# ---------------------------------------------------------------- serving calls
@pytest.fixture(scope="module")
def models():
    torch.manual_seed(0)
    out = {}
    for prec in ("bf16", "fp32"):
        m = hk.KeypointsGauss(4, precision=prec)
        out[prec] = m.cuda().eval()
    return out


def _images(seed, B=2, H=96, W=128):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(B, 3, H, W, generator=g).cuda()
    x8 = (torch.rand(B, H, W, 3, generator=g) * 255).to(torch.uint8).cuda()
    return x, x8


@pytest.mark.parametrize("prec", ["bf16", "fp32"])
def test_model_peaks_equals_eager_decode_of_forward(models, prec):
    m = models[prec]
    x, x8 = _images(1)
    for inp in (x, x8):
        for slot in (0, 1):
            heat = m(inp)
            thr = float(heat.median())
            got = [t.clone() for t in m.peaks(inp, max_peaks=32, threshold=thr, min_distance=3, slot=slot)]
            want = ops.peak_decode(heat, 32, thr, 3)
            assert all(torch.equal(a, b) for a, b in zip(got, want)), (inp.dtype, slot)
            assert int(got[2].max()) > 1


def test_model_peaks_recaptures_on_parameter_change(models):
    m = models["bf16"]
    x, _ = _images(2)
    heat = m(x)
    thr = float(heat.median())
    for N, t, r in ((4, thr, 2), (16, thr, 2), (16, thr + 1e-3, 2), (16, thr + 1e-3, 5)):
        got = m.peaks(x, max_peaks=N, threshold=t, min_distance=r)
        want = ops.peak_decode(heat, N, t, r)
        assert all(torch.equal(a, b) for a, b in zip(got, want)), (N, t, r)


def test_keypoints_interleaved_with_peaks(models):
    m = models["bf16"]
    x, _ = _images(3)
    heat = m(x)
    want_yx, want_max = ops.argmax_decode(heat, want_max=True)
    for _ in range(2):
        yx, mx = m.keypoints(x)
        assert torch.equal(yx, want_yx) and torch.equal(mx, want_max)
        got = m.peaks(x, max_peaks=8, threshold=0.0, min_distance=4)
        assert torch.equal(got[0][..., 0, :], want_yx) and torch.equal(got[1][..., 0], want_max)


def test_model_peaks_rejects_bad_arguments(models):
    x, _ = _images(4)
    for kw in (dict(max_peaks=0), dict(min_distance=17), dict(threshold=float("nan"))):
        with pytest.raises(ValueError):
            models["bf16"].peaks(x, **kw)


def test_prediction_peaks_numpy_and_cuda_agree(models):
    pred = Prediction(models["bf16"], 4, 96, 128, use_cuda=True)
    heat = torch.rand((2, 4, 96, 128), device="cuda", generator=_gen(8))
    a = pred.peaks(heat, max_peaks=16, threshold=0.5, min_distance=4)
    b = pred.peaks(heat.cpu().numpy(), max_peaks=16, threshold=0.5, min_distance=4)
    assert [t.dtype for t in a] == [np.int64, np.float32, np.int64] and a[0].shape == (2, 4, 16, 2)
    assert all(np.array_equal(u, v) for u, v in zip(a, b))
    ryx, rscore, rcount = peak_decode_ref(heat.cpu().numpy(), 16, 0.5, 4)
    assert np.array_equal(a[0], ryx) and np.array_equal(a[1], rscore) and np.array_equal(a[2], rcount)
