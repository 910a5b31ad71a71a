"""Host side of Qwen2.5-VL video scoring (no GPU): the frame sampling and sizing restated from qwen_vl_utils, the processor's
temporal-patch layout against the installed transformers, the torchvision-policy tap tables of the device kernel replayed on the CPU
against torchvision, the cv2 decoder, and the routing of video paths through Score."""
import numpy as np
import pytest
import torch

from t2v_metrics_b200.models.vqascore_models import qwen_utils as qu


# ---------------------------------------------------------------------------------------------- sampling and sizing
def test_smart_nframes_hand_computed():
    # 5 s at 24 fps sampled at 8 fps: 120 / 24 * 8 = 40
    assert qu.smart_nframes(120, 24.0, 8.0) == 40
    # fps="dynamic" -> FPS = 2.0: 120 / 24 * 2 = 10
    assert qu.smart_nframes(120, 24.0, qu.FPS) == 10
    # a rate above the clip's own: clamped to total (floor2(min(768, 31)) = 30), then floor2 -> 30
    assert qu.smart_nframes(31, 10.0, 100.0) == 30
    # odd frame count, low rate: 9 / 30 * 2 = 0.6 -> raised to FPS_MIN_FRAMES = 4
    assert qu.smart_nframes(9, 30.0, 2.0) == 4
    # a clip shorter than 4 frames: min(max(x, 4), floor2(3) = 2) = 2, min(., 3) = 2
    assert qu.smart_nframes(3, 30.0, 2.0) == 2
    # 1 frame: floor2(min(1, ...)) = 0 < FRAME_FACTOR -> raises
    with pytest.raises(ValueError):
        qu.smart_nframes(1, 30.0, 2.0)
    # long clip: FPS_MAX_FRAMES caps it
    assert qu.smart_nframes(100000, 30.0, 8.0) == 768


def test_sample_indices_and_fps():
    assert qu.sample_frame_indices(120, 40)[:4] == [0, 3, 6, 9] and qu.sample_frame_indices(120, 40)[-1] == 119
    idx = qu.sample_frame_indices(9, 4)                     # linspace(0, 8, 4) = 0, 2.667, 5.333, 8
    assert idx == [0, 3, 5, 8]
    assert qu.sample_frame_indices(3, 2) == [0, 2]
    assert qu.video_sample_fps(40, 120, 24.0) == pytest.approx(8.0)
    assert qu.video_sample_fps(4, 9, 30.0) == pytest.approx(4 / 9 * 30)
    assert qu.second_per_grid(2) == 2 / 24 and qu.second_per_grid(2, 8.0) == 0.25


def test_video_pixel_budget_and_frame_size():
    # VIDEO_TOTAL_PIXELS / nframes * 2 is far above VIDEO_MAX_PIXELS for short clips: min(768*784, ...) then the reference's 360*420
    assert qu.video_max_pixels(40) == 360 * 420
    assert qu.video_max_pixels(40, None) == 768 * 28 * 28
    # many frames: the total budget bites, floored at int(VIDEO_MIN_PIXELS * 1.05)
    assert qu.video_max_pixels(768, None) == pytest.approx(max(min(768 * 784, int(128000 * 784 * 0.9) / 768 * 2), int(128 * 784 * 1.05)))
    assert qu.video_max_pixels(100000, None) == int(128 * 784 * 1.05)
    # 640x360 at 360*420: round -> 364 x 644 > 151200 -> beta = sqrt(230400 / 151200), floor -> 280 x 504 (grid 20 x 36)
    assert qu.video_frame_size(360, 640, 40) == (280, 504)
    # small frames are raised to VIDEO_MIN_PIXELS: 100x150 -> beta = sqrt(100352 / 15000) -> ceil -> 280 x 392
    assert qu.video_frame_size(100, 150, 4) == (280, 392)


# ---------------------------------------------------------------------------------------------- processor layout
@pytest.mark.parametrize("frames,hw", [(4, (56, 84)), (6, (112, 56)), (2, (28 * 4, 28 * 3))])
def test_video_to_patches_matches_transformers(frames, hw):
    from transformers.models.qwen2_vl.video_processing_qwen2_vl import Qwen2VLVideoProcessor
    rng = np.random.default_rng(frames)
    v = rng.integers(0, 256, (frames, *hw, 3), dtype=np.uint8)
    rows, grid = qu.qwen_video_to_patches(v)
    proc = Qwen2VLVideoProcessor(do_resize=False)
    out = proc(videos=[torch.from_numpy(v).permute(0, 3, 1, 2)], return_tensors="pt")
    assert tuple(out["video_grid_thw"][0].tolist()) == grid == (frames // 2, hw[0] // 14, hw[1] // 14)
    ref = out["pixel_values_videos"].float()
    assert ref.shape == rows.shape
    # same tolerance as the still-image processor test: fp32 rescale/normalise orders differ in the last bits
    torch.testing.assert_close(rows, ref, rtol=1e-5, atol=1e-5)


def test_odd_frame_stack_repeats_last_frame():
    rng = np.random.default_rng(1)
    v = rng.integers(0, 256, (3, 56, 56, 3), dtype=np.uint8)
    stacked = qu.pil_resize_frames(v)
    assert stacked.shape[0] == 4 and np.array_equal(stacked[3], stacked[2])
    a, ga = qu.qwen_video_to_patches(v)
    b, gb = qu.qwen_video_to_patches(stacked)
    assert ga == gb == (2, 4, 4) and torch.equal(a, b)


def test_second_per_grid_matches_processor():
    from transformers import Qwen2_5_VLProcessor
    from transformers.models.qwen2_vl.video_processing_qwen2_vl import Qwen2VLVideoProcessor
    from transformers.models.qwen2_vl.image_processing_qwen2_vl import Qwen2VLImageProcessor
    tok = _tiny_tokenizer()
    if tok is None:
        pytest.skip("no tokenizer to build a Qwen2_5_VLProcessor offline")
    proc = Qwen2_5_VLProcessor(image_processor=Qwen2VLImageProcessor(), tokenizer=tok, video_processor=Qwen2VLVideoProcessor())
    v = torch.zeros(4, 3, 56, 56, dtype=torch.uint8)
    # the reference's call: pre-sampled frames plus the reader's rate as `fps` (frame stacks: 2.0; files: nframes / total * rate)
    for fps in (2.0, 8.0, 24 * 40 / 120):
        out = proc(text=["<|vision_start|><|video_pad|><|vision_end|>"], videos=[v], fps=fps, do_resize=False, return_tensors="pt")
        assert float(out["second_per_grid_ts"][0]) == pytest.approx(qu.second_per_grid(2), rel=1e-6)


def _tiny_tokenizer():
    try:
        from transformers import PreTrainedTokenizerFast
        from tokenizers import Tokenizer, models, pre_tokenizers
    except ImportError:
        return None
    specials = ["<|im_start|>", "<|im_end|>", "<|vision_start|>", "<|vision_end|>", "<|image_pad|>", "<|video_pad|>", "<unk>"]
    vocab = {t: i for i, t in enumerate(specials + list("abcdefghijklmnopqrstuvwxyz "))}
    t = Tokenizer(models.WordLevel(vocab, unk_token="<unk>"))
    t.pre_tokenizer = pre_tokenizers.Split("", "isolated")
    tok = PreTrainedTokenizerFast(tokenizer_object=t, unk_token="<unk>", additional_special_tokens=specials[:6])
    tok.image_token, tok.video_token = "<|image_pad|>", "<|video_pad|>"
    return tok


# ---------------------------------------------------------------------------------------------- torchvision-policy replay
def _replay_axis(x: np.ndarray, bounds, taps, fma: bool) -> np.ndarray:
    """One pass of the kernel's torchvision policy along the last axis: acc = 0; acc = fma(px, w, acc) or acc + round(px * w),
    sequentially over the window (zero taps past the window add exact zeros)."""
    out_n, ks = taps.shape
    n = x.shape[-1]
    acc = np.zeros(x.shape[:-1] + (out_n,), np.float32)
    for j in range(ks):
        idx = np.minimum(bounds[:, 0] + j, n - 1)
        w = np.where(j < bounds[:, 1], taps[:, j], 0).astype(np.float32)
        px = x[..., idx]
        if fma:
            # fp32 fma: the product is exact in fp64; the fp64 sum rounded once more to fp32 can differ from a true fma only at
            # double-rounding ties, far rarer than the fp32 ties this test bounds
            acc = (acc.astype(np.float64) + px.astype(np.float64) * w.astype(np.float64)).astype(np.float32)
        else:
            acc = (acc + (px * w).astype(np.float32)).astype(np.float32)
    return acc


def replay_torchvision_resize(frames_u8: np.ndarray, h: int, w: int) -> np.ndarray:
    from t2v_metrics_b200.engine import resample_table_tv
    x = frames_u8.astype(np.float32).transpose(0, 3, 1, 2)           # T, C, H, W
    bh, th, fh = resample_table_tv(x.shape[2], h)
    bw, tw, fw = resample_table_tv(x.shape[3], w)
    y = _replay_axis(x, bw.numpy(), tw.numpy(), fw)                   # width first
    y = _replay_axis(y.transpose(0, 1, 3, 2), bh.numpy(), th.numpy(), fh).transpose(0, 1, 3, 2)
    return np.rint(np.clip(y, 0, 255)).astype(np.uint8).transpose(0, 2, 3, 1)


# measured with torch 2.11 (x86-64 CPU build, AVX512 kernels): 1 value off by one grey level in 776160 on 480x640 -> 308x420, none on the
# other shapes; the documented bound is 1 grey level on < 0.01 % of values
TIE_BOUND = 1e-4


@pytest.mark.parametrize("src,dst", [((360, 640), (280, 504)), ((480, 640), (308, 420)), ((100, 150), (224, 336)),
                                     ((57, 91), (56, 84)), ((90, 61), (336, 224)), ((123, 77), (84, 140)), ((224, 224), (224, 224))])
def test_torchvision_policy_replay_matches_torchvision(src, dst):
    pytest.importorskip("t2v_metrics_b200._lib").load()
    tvf = pytest.importorskip("torchvision.transforms.functional")
    from torchvision.transforms import InterpolationMode
    rng = np.random.default_rng(src[0] * 7 + dst[1])
    v = rng.integers(0, 256, (2, *src, 3), dtype=np.uint8)
    ref = tvf.resize(torch.from_numpy(v).permute(0, 3, 1, 2), list(dst), interpolation=InterpolationMode.BICUBIC, antialias=True)
    ref = ref.permute(0, 2, 3, 1).numpy()
    got = replay_torchvision_resize(v, *dst)
    diff = np.abs(got.astype(np.int32) - ref.astype(np.int32))
    frac = float((diff > 0).mean())
    print(f"\n[tv replay {src}->{dst}] mismatching {int((diff > 0).sum())} / {diff.size} ({frac:.2e}), max {int(diff.max())}")
    assert diff.max() <= 1 and frac < TIE_BOUND
    # the host helper (what fetch_video computes) is torchvision's result too
    host = qu.torchvision_resize_u8(torch.from_numpy(v), *dst).numpy()
    assert np.array_equal(host, ref)


def test_tv_tap_table_shape_and_normalisation():
    pytest.importorskip("t2v_metrics_b200._lib").load()
    from t2v_metrics_b200.engine import resample_table_tv
    b, t, fma = resample_table_tv(640, 504)
    assert b.shape == (504, 2) and t.shape[1] == 7 and not fma
    assert torch.all(b[:, 1] <= 7) and torch.all(b[:, 0] >= 0) and torch.all(b[:, 0] + b[:, 1] <= 640)
    assert torch.allclose(t.sum(1), torch.ones(504), atol=1e-6)
    _, t2, fma2 = resample_table_tv(150, 336)
    assert fma2 and t2.shape[1] == 5


def test_video_plan_grids():
    pytest.importorskip("t2v_metrics_b200._lib").load()
    from t2v_metrics_b200 import _lib
    from t2v_metrics_b200.engine import qwen_video_preprocess_plan
    grids, rows, wsb = qwen_video_preprocess_plan([(40, 360, 640), (3, 56, 56), (16, 224, 224)],
                                                  [_lib.VQA_RESAMPLE_TORCHVISION, _lib.VQA_RESAMPLE_PIL, _lib.VQA_RESAMPLE_PIL],
                                                  [qu.VIDEO_MIN_PIXELS, qu.QWEN_VL_UTILS_MIN_PIXELS, qu.QWEN_VL_UTILS_MIN_PIXELS],
                                                  [qu.REFERENCE_VIDEO_MAX_PIXELS, qu.QWEN_VL_UTILS_MAX_PIXELS, qu.QWEN_VL_UTILS_MAX_PIXELS])
    assert grids == [(20, 20, 36), (2, 4, 4), (8, 16, 16)]
    assert rows == 20 * 20 * 36 + 2 * 16 + 8 * 256 and wsb > 0


# ---------------------------------------------------------------------------------------------- cv2 decode
def test_cv2_round_trip(tmp_path):
    cv2 = pytest.importorskip("cv2")
    path = str(tmp_path / "clip.avi")
    wr = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"MJPG"), 24.0, (64, 48))
    if not wr.isOpened():
        pytest.skip("this OpenCV build cannot write MJPG")
    for i in range(30):
        f = np.zeros((48, 64, 3), np.uint8)
        f[:, :, 2] = i * 8              # BGR: frame number in the red channel
        wr.write(f)
    wr.release()
    frames, sample_fps, idx = qu.decode_video_cv2(path, 8.0)
    n = qu.smart_nframes(30, 24.0, 8.0)                 # 30 / 24 * 8 = 10
    assert n == 10 and frames.shape == (10, 48, 64, 3) and idx == qu.sample_frame_indices(30, 10)
    assert sample_fps == pytest.approx(10 / 30 * 24.0)
    red = frames[..., 0].reshape(10, -1).mean(1)        # RGB after the conversion
    assert np.all(np.abs(red - np.array(idx) * 8) < 4)
    frames_d, fps_d, idx_d = qu.decode_video_cv2(path, "dynamic")
    assert len(idx_d) == qu.smart_nframes(30, 24.0, qu.FPS) == 4


# ---------------------------------------------------------------------------------------------- Score routing
class _StubPlugin:
    def __init__(self, video_mode):
        self.video_mode = video_mode
        self.calls = []

    def forward(self, images, texts, **kw):
        self.calls.append((list(images), list(texts), kw))
        return torch.tensor([float(len(i) + len(t)) for i, t in zip(images, texts)])


def _score(video_mode):
    from t2v_metrics_b200.score import Score

    class S(Score):
        def prepare_scoremodel(self, model, device, cache_dir, **kwargs):
            return _StubPlugin(video_mode)

        def list_all_models(self):
            return ["stub"]
    return S("stub", device="cpu")


def test_score_routes_videos_to_direct_plugin():
    s = _score("direct")
    out = s(images=["a.mp4", "b.npy", "c.png"], texts=["x", "yy"], fps="dynamic")
    assert out.shape == (3, 2)
    imgs, texts, kw = s.model.calls[0]
    assert imgs == ["a.mp4", "a.mp4", "b.npy", "b.npy", "c.png", "c.png"] and kw == {"fps": "dynamic"}
    with pytest.raises(NotImplementedError):
        _score("concat")(images=["a.mp4"], texts=["x"])


def test_batch_forward_videos():
    s = _score("direct")
    ds = [{"videos": [f"v{i}.mp4", f"w{i}.avi"], "texts": ["t", "uu", "vvv"]} for i in range(5)]
    out = s.batch_forward(ds, batch_size=2)
    assert out.shape == (5, 2, 3)
    assert float(out[0, 0, 1]) == len("v0.mp4") + 2 and float(out[4, 1, 2]) == len("w4.avi") + 3
    with pytest.raises(NotImplementedError):
        _score("concat").batch_forward(ds)
