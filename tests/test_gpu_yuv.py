"""GPU: YUV 4:2:0 input.  k_yuv420_to_bgr (apse_cvt_yuv420_bgr) equals cv2.cvtColor(COLOR_YUV2BGR_{NV12,NV21,I420,YV12}) and
the CPU restatement tools/yuv_reference.py byte for byte (every (Y, U, V) triple, odd h/2, widths off the 16-byte vector path, unaligned buffers, batches whose
offsets pass 2^31); the drop-in cvtColor codes; and the host-frame pipeline fed with YUV batches gives the results of the same
frames converted to BGR on the host."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

LAYOUTS = ("nv12", "nv21", "i420", "yv12")
SIZES = ((3840, 2160), (1920, 1082), (1922, 1080), (66, 6), (2, 2))


def _code(cv2, layout):
    return {"nv12": cv2.COLOR_YUV2BGR_NV12, "nv21": cv2.COLOR_YUV2BGR_NV21, "i420": cv2.COLOR_YUV2BGR_I420,
            "yv12": cv2.COLOR_YUV2BGR_YV12}[layout]


@pytest.fixture(scope="module")
def eng():
    from apse_uav_b200 import Engine
    e = Engine(0, 64, 64, 1)   # the conversion uses no context scratch: frames larger than max_w x max_h are fine
    yield e
    e.close()


@pytest.mark.parametrize("layout", LAYOUTS)
def test_all_triples(eng, layout):
    cv2 = pytest.importorskip("cv2")
    from tools import synth, yuv_reference
    yuv = synth.yuv420_all_triples(layout)
    got = eng.cvt_yuv420(yuv, layout).cpu().numpy()
    assert np.array_equal(got, cv2.cvtColor(yuv, _code(cv2, layout)))
    assert np.array_equal(got, yuv_reference.yuv420_to_bgr(yuv, layout))


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("size", SIZES, ids=[f"{w}x{h}" for w, h in SIZES])
def test_frame_sizes(eng, layout, size):
    cv2 = pytest.importorskip("cv2")
    w, h = size
    yuv = np.random.default_rng(w + 3 * h).integers(0, 256, (h * 3 // 2, w), dtype=np.uint8)
    assert np.array_equal(eng.cvt_yuv420(yuv, layout).cpu().numpy(), cv2.cvtColor(yuv, _code(cv2, layout)))


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("shift", [(1, 0), (0, 1), (1, 1)], ids=["src+1", "dst+1", "both+1"])
def test_unaligned_buffers(eng, layout, shift):
    """source / destination one byte past their alignment: the 4K frame takes the scalar path and still matches"""
    cv2 = pytest.importorskip("cv2")
    import torch
    w, h = 3840, 2160
    yuv = np.random.default_rng(11).integers(0, 256, (h * 3 // 2, w), dtype=np.uint8)
    sbuf = torch.empty(yuv.size + 16, dtype=torch.uint8, device="cuda")
    dbuf = torch.empty(w * h * 3 + 16, dtype=torch.uint8, device="cuda")
    src = sbuf[shift[0]:shift[0] + yuv.size].view(h * 3 // 2, w)
    src.copy_(torch.from_numpy(yuv))
    dst = dbuf[shift[1]:shift[1] + w * h * 3].view(h, w, 3)
    eng.cvt_yuv420(src, layout, out=dst)
    assert np.array_equal(dst.cpu().numpy(), cv2.cvtColor(yuv, _code(cv2, layout)))


@pytest.mark.parametrize("layout", LAYOUTS)
def test_batch_equals_single_frames(eng, layout):
    """a 4K batch of 21 frames: every frame equals its single-frame conversion and cv2"""
    cv2 = pytest.importorskip("cv2")
    import torch
    w, h, n = 3840, 2160, 21
    g = torch.Generator(device="cuda").manual_seed(5)
    batch = torch.randint(0, 256, (n, h * 3 // 2, w), dtype=torch.uint8, device="cuda", generator=g)
    out = eng.cvt_yuv420(batch, layout)
    assert tuple(out.shape) == (n, h, w, 3)
    for i in range(n):
        assert torch.equal(out[i], eng.cvt_yuv420(batch[i], layout)), i
    for i in (0, n - 1):
        assert np.array_equal(out[i].cpu().numpy(), cv2.cvtColor(batch[i].cpu().numpy(), _code(cv2, layout)))


def test_batch_offsets_past_2_31(eng):
    """90 4K frames: the output of frames 87 and later starts beyond 2^31 bytes"""
    cv2 = pytest.importorskip("cv2")
    import torch
    w, h, n = 3840, 2160, 90
    assert 86 * w * h * 3 < 2 ** 31 < 87 * w * h * 3
    g = torch.Generator(device="cuda").manual_seed(9)
    base = torch.randint(0, 256, (6, h * 3 // 2, w), dtype=torch.uint8, device="cuda", generator=g)
    batch = base.repeat(15, 1, 1)
    batch[:, 0, 0] = torch.arange(n, dtype=torch.uint8, device="cuda")   # every frame distinct
    for layout in ("nv12", "i420"):
        out = eng.cvt_yuv420(batch, layout)
        for i in (0, 45, 86, 87, 88, 89):
            assert np.array_equal(out[i].cpu().numpy(), cv2.cvtColor(batch[i].cpu().numpy(), _code(cv2, layout))), (layout, i)
        del out
        torch.cuda.empty_cache()


def test_argument_errors(eng):
    import torch
    from apse_uav_b200 import ApseError
    good = torch.zeros((6, 4), dtype=torch.uint8, device="cuda")
    out = torch.empty((4, 4, 3), dtype=torch.uint8, device="cuda")
    with pytest.raises(ApseError):   # odd width
        eng.cvt_yuv420(torch.zeros((6, 5), dtype=torch.uint8, device="cuda"), "nv12")
    with pytest.raises(ApseError):   # unknown layout name
        eng.cvt_yuv420(good, "yuy2")
    with pytest.raises(ApseError):   # rows not divisible by 3
        eng.cvt_yuv420(torch.zeros((7, 4), dtype=torch.uint8, device="cuda"), "nv12")
    lib, st = eng.lib, eng._stream()
    assert lib.apse_cvt_yuv420_bgr(eng.h, good.data_ptr(), 4, 3, 1, 0, out.data_ptr(), st) == -1   # odd height
    assert lib.apse_cvt_yuv420_bgr(eng.h, good.data_ptr(), 5, 4, 1, 0, out.data_ptr(), st) == -1   # odd width
    assert lib.apse_cvt_yuv420_bgr(eng.h, good.data_ptr(), 4, 4, 1, 4, out.data_ptr(), st) == -1   # unknown layout
    assert lib.apse_cvt_yuv420_bgr(eng.h, good.data_ptr(), 4, 4, 1, -1, out.data_ptr(), st) == -1
    assert lib.apse_cvt_yuv420_bgr(eng.h, good.data_ptr(), 4, 4, 0, 0, out.data_ptr(), st) == -1   # empty batch
    assert lib.apse_cvt_yuv420_bgr(eng.h, None, 4, 4, 1, 0, out.data_ptr(), st) == -1
    assert lib.apse_cvt_yuv420_bgr(eng.h, good.data_ptr(), 4, 4, 1, 0, None, st) == -1
    assert lib.apse_cvt_yuv420_bgr(eng.h, good.data_ptr(), 4, 4, 1, 0, out.data_ptr(), st) == 0


def test_dropin_cvtcolor():
    cv2 = pytest.importorskip("cv2")
    import torch
    import apse_uav_b200 as A
    yuv = np.random.default_rng(2).integers(0, 256, (1082 * 3 // 2, 1920), dtype=np.uint8)
    for code in (A.COLOR_YUV2BGR_NV12, A.COLOR_YUV2BGR_NV21, A.COLOR_YUV2BGR_I420, A.COLOR_YUV2BGR_IYUV, A.COLOR_YUV2BGR_YV12):
        want = cv2.cvtColor(yuv, code)
        got = A.cvtColor(yuv, code)
        assert isinstance(got, np.ndarray) and np.array_equal(got, want), code
        got_t = A.cvtColor(torch.from_numpy(yuv).cuda(), code)
        assert isinstance(got_t, torch.Tensor) and got_t.is_cuda and np.array_equal(got_t.cpu().numpy(), want), code
    assert (A.COLOR_YUV2BGR_NV12, A.COLOR_YUV2BGR_NV21, A.COLOR_YUV2BGR_YV12, A.COLOR_YUV2BGR_I420, A.COLOR_YUV2BGR_IYUV) == \
        (cv2.COLOR_YUV2BGR_NV12, cv2.COLOR_YUV2BGR_NV21, cv2.COLOR_YUV2BGR_YV12, cv2.COLOR_YUV2BGR_I420, cv2.COLOR_YUV2BGR_IYUV)
    for code in (cv2.COLOR_YUV2RGB_NV12, cv2.COLOR_YUV2GRAY_420, 40):
        with pytest.raises(A.ApseError):
            A.cvtColor(yuv, code)


# ---- the host-frame pipeline fed with YUV batches ------------------------------------------------------------------------
@pytest.fixture(scope="module")
def events_yuv(dictionary):
    """the 64-frame events sequence in every layout (derived from cv2's BGR -> I420 planes) and the same frames converted back
    to BGR on the host"""
    cv2 = pytest.importorskip("cv2")
    from conftest import golden_csv, golden_events
    from tools import synth
    g, _ = golden_csv("sequence_4k_events.json")
    frames = list(synth.make_sequence(dictionary.bytesList, g["base_seed"], g["n_frames"], leds=g["leds"], events=golden_events(g)))
    yuv = {l: np.stack([synth.bgr_to_yuv420(f, l) for f in frames]) for l in LAYOUTS}
    bgr = np.stack([cv2.cvtColor(f, cv2.COLOR_YUV2BGR_I420) for f in yuv["i420"]])
    for l in LAYOUTS:   # the four layouts carry the same pixels
        assert np.array_equal(cv2.cvtColor(yuv[l][-1], _code(cv2, l)), bgr[-1])
    return yuv, bgr


@pytest.fixture(scope="module")
def pipe3(camera, lut, dictionary, ref_params):
    import apse_uav_b200 as A
    K, D = camera
    p = A.Pipeline(K, D, (3840, 2160), lut, dictionary, ref_params, max_batch=6, max_markers=64, streams=3)
    yield p
    p.close()


def _pinned_batches(a, b):
    import torch
    t = torch.from_numpy(a).pin_memory()
    return [t[i:i + b] for i in range(0, len(a), b)]


@pytest.mark.parametrize("leds", [False, True])
def test_sequence_host_yuv_equals_host_converted_bgr(pipe3, events_yuv, leds):
    """shard.run_sequence_host(layout=...) on YUV batches (64 frames, max_batch 6: a last batch of 4) gives the rows and the CSV
    text of run_sequence_host on the host-converted BGR batches; Pipeline.run_host_stream gives the same per-frame results"""
    from apse_uav_b200 import shard, sequence
    yuv, bgr = events_yuv
    n = len(bgr)
    want = shard.run_sequence_host(pipe3, _pinned_batches(bgr, 6), n, leds=leds, as_rows=True)
    want_csv = sequence.rows_to_csv(want)
    for layout in LAYOUTS:
        rows = shard.run_sequence_host(pipe3, _pinned_batches(yuv[layout], 6), n, leds=leds, as_rows=True, layout=layout)
        assert rows.dtype == want.dtype and rows.tobytes() == want.tobytes(), layout
        assert sequence.rows_to_csv(rows) == want_csv, layout
    if leds:
        return
    ref = list(pipe3.run_host_stream(_pinned_batches(bgr, 6)))
    for layout in ("nv12", "yv12"):
        got = list(pipe3.run_host_stream(_pinned_batches(yuv[layout], 6), layout=layout))
        assert len(got) == len(ref)
        for a, b in zip(got, ref):
            for k in ("n", "ids", "corners", "rvec", "tvec"):
                assert np.array_equal(a[k], b[k]), (layout, k)


def test_host_stream_nv12_equals_run_batch(pipe3, events_yuv):
    """Pipeline.run_host_stream(layout="nv12") equals run_batch on the frames converted on the host"""
    import torch
    yuv, bgr = events_yuv
    frames = bgr[:14]
    got = list(pipe3.run_host_stream(_pinned_batches(yuv["nv12"][:14], 6), layout="nv12"))
    assert [len(r["n"]) for r in got] == [6, 6, 2]
    for j, r in enumerate(got):
        ref = pipe3.to_host(pipe3.run_batch(torch.from_numpy(frames[6 * j:6 * j + 6]).cuda()))
        for k in ("n", "ids", "corners", "rvec", "tvec"):
            assert np.array_equal(r[k], ref[k]), (j, k)
    assert int(sum(r["n"].sum() for r in got)) > 0


def test_host_batches_of_the_wrong_shape_raise(pipe3, events_yuv):
    import torch
    from apse_uav_b200 import ApseError
    _, bgr = events_yuv
    with pytest.raises(ApseError):   # a BGR batch handed in as NV12
        list(pipe3.run_host_stream([torch.from_numpy(bgr[:2]).pin_memory()], layout="nv12"))
    torch.cuda.synchronize()
