"""Qwen2.5-VL video scoring on the GPU: the device pre-processing kernel against the host pipeline (PIL frame stacks bit for bit,
torchvision-policy decoded frames up to fp32 ties), the plugin on a mix of a frame stack, a video file and an image against the oracle,
and the engine at full 7B width on a realistic video length against the real HF model."""
import dataclasses
import gc

import numpy as np
import pytest
import torch

from oracle import qwen25vl_oracle as qo
from t2v_metrics_b200.models.vqascore_models import qwen_utils as qu

pytestmark = pytest.mark.gpu

TINY = dict(hidden=256, heads=2, kv_heads=1, mrope_section=(16, 24, 24))
TIE_BOUND = 1e-4            # torchvision policy: at most 1 grey level on fewer than 0.01 % of values


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    return torch.device("cuda:0")


def _lut_steps(got: torch.Tensor, ref: torch.Tensor) -> torch.Tensor:
    """Grey-level distance of two normalised patch-row tensors (columns (c, t, py, px)): |diff| * 255 * std[c]."""
    std = torch.tensor(qu.OPENAI_CLIP_STD).repeat_interleave(got.shape[1] // 3)
    return ((got.cpu() - ref) * 255.0 * std).abs()


@pytest.mark.parametrize("frames,hw", [(4, (56, 84)), (5, (60, 80)), (7, (123, 200)), (16, (224, 224))])
def test_video_kernel_pil_frame_stacks_bit_identical(dev, frames, hw):
    from t2v_metrics_b200 import _lib
    from t2v_metrics_b200.engine import qwen_video_preprocess_u8
    rng = np.random.default_rng(frames * 1000 + hw[0])
    vids = [rng.integers(0, 256, (frames, *hw, 3), dtype=np.uint8), rng.integers(0, 256, (3, 40, 52, 3), dtype=np.uint8)]
    got, grids = qwen_video_preprocess_u8([torch.from_numpy(v) for v in vids], [_lib.VQA_RESAMPLE_PIL] * 2, dev,
                                          [qu.QWEN_VL_UTILS_MIN_PIXELS] * 2, [qu.QWEN_VL_UTILS_MAX_PIXELS] * 2)
    torch.cuda.synchronize()
    refs = [qu.qwen_video_to_patches(qu.pil_resize_frames(v)) for v in vids]
    assert grids == [g for _, g in refs]
    assert torch.equal(got.cpu(), torch.cat([r for r, _ in refs]))
    bf, _ = qwen_video_preprocess_u8([torch.from_numpy(v) for v in vids], [_lib.VQA_RESAMPLE_PIL] * 2, dev,
                                     [qu.QWEN_VL_UTILS_MIN_PIXELS] * 2, [qu.QWEN_VL_UTILS_MAX_PIXELS] * 2, out_dtype=torch.bfloat16)
    assert torch.equal(bf.cpu(), got.cpu().to(torch.bfloat16))


@pytest.mark.parametrize("frames,hw", [(40, (360, 640)), (6, (480, 640)), (4, (100, 150)), (8, (57, 91))])
def test_video_kernel_torchvision_policy(dev, frames, hw):
    from torchvision.transforms import InterpolationMode
    import torchvision.transforms.functional as tvf
    from t2v_metrics_b200 import _lib
    from t2v_metrics_b200.engine import qwen_video_preprocess_u8
    rng = np.random.default_rng(frames + hw[1])
    v = rng.integers(0, 256, (frames, *hw, 3), dtype=np.uint8)
    mx = int(qu.video_max_pixels(frames))
    rh, rw = qu.smart_resize(*hw, 28, qu.VIDEO_MIN_PIXELS, mx)
    got, grids = qwen_video_preprocess_u8([torch.from_numpy(v)], [_lib.VQA_RESAMPLE_TORCHVISION], dev, [qu.VIDEO_MIN_PIXELS], [mx])
    torch.cuda.synchronize()
    host, hgrid = qu.qwen_video_to_patches(qu.torchvision_resize_u8(torch.from_numpy(v), rh, rw))
    tv = tvf.resize(torch.from_numpy(v).permute(0, 3, 1, 2), [rh, rw], interpolation=InterpolationMode.BICUBIC, antialias=True)
    direct, _ = qu.qwen_video_to_patches(tv.permute(0, 2, 3, 1).numpy())
    assert grids == [hgrid]
    for name, ref in (("host pipeline", host), ("torchvision", direct)):
        steps = _lut_steps(got, ref)
        frac = float((steps > 0.5).float().mean())
        print(f"\n[tv kernel {frames}x{hw} -> {rh}x{rw} vs {name}] values off by one grey level: {int((steps > 0.5).sum())} "
              f"({frac:.2e}); max {float(steps.max()):.3f} levels")
        assert float(steps.max()) < 1.01 and frac < TIE_BOUND


class FakeTokenizer:
    """Character-level ids below the tiny config's vision ids; enough for build_prompt_ids and the answer token."""
    eos_token_id, bos_token_id, pad_token_id = 599, None, 598

    def encode(self, s, add_special_tokens=False):
        return [1 + (ord(c) % 500) for c in s]

    def decode(self, ids):
        return "".join(chr(i - 1) for i in ids)


def _write_video(path_mp4: str, frames: np.ndarray, fps: float) -> str:
    cv2 = pytest.importorskip("cv2")
    h, w = frames.shape[1:3]
    for path, code in ((path_mp4, "mp4v"), (path_mp4[:-4] + ".avi", "MJPG")):
        wr = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*code), fps, (w, h))
        if wr.isOpened():
            for f in frames:
                wr.write(cv2.cvtColor(f, cv2.COLOR_RGB2BGR))
            wr.release()
            return path
    pytest.skip("this OpenCV build can write neither mp4v nor MJPG")


def test_plugin_mixed_video_stack_image_matches_oracle(dev, tmp_path):
    from PIL import Image
    from t2v_metrics_b200.config import Qwen25VLConfig
    from t2v_metrics_b200.models.vqascore_models.qwen2vl_model import Qwen2VLModel
    ocfg = qo.Qwen25VLConfig.tiny(**TINY)
    sd = qo.make_synthetic_state_dict(ocfg, seed=4)
    fields = {f.name for f in dataclasses.fields(Qwen25VLConfig)}
    cfg = Qwen25VLConfig(**{k: v for k, v in dataclasses.asdict(ocfg).items() if k in fields})
    rng = np.random.default_rng(7)
    stack = rng.integers(0, 256, (5, 60, 80, 3), dtype=np.uint8)                     # odd count: last frame repeated
    np.save(tmp_path / "stack.npy", stack)
    clip = np.repeat(np.repeat(rng.integers(0, 256, (12, 12, 16, 3), dtype=np.uint8), 4, 1), 4, 2)   # 12 frames 48x64, smooth
    vpath = _write_video(str(tmp_path / "clip.mp4"), clip, 24.0)
    img = rng.integers(0, 256, (70, 90, 3), dtype=np.uint8)
    Image.fromarray(img).save(tmp_path / "img.png")
    paths = [vpath, str(tmp_path / "stack.npy"), str(tmp_path / "img.png")]
    texts = ["a red car", "two dogs"]
    model = Qwen2VLModel(device="cuda", tokenizer=FakeTokenizer(), state_dict={k: v.clone() for k, v in sd.items()}, config=cfg,
                         repetition_penalty=1.0)
    pair_paths = [p for p in paths for _ in texts]
    pair_texts = [t for _ in paths for t in texts]
    got = model.forward(pair_paths, pair_texts)
    # the host pipeline: what the reference computes for each input
    frames, _, _ = qu.decode_video_cv2(vpath, 8.0)
    rh, rw = qu.video_frame_size(*frames.shape[1:3], len(frames))
    rows_v, g_v = qu.qwen_video_to_patches(qu.torchvision_resize_u8(torch.from_numpy(frames), rh, rw))
    rows_s, g_s = qu.qwen_video_to_patches(qu.pil_resize_frames(stack))
    rows_i, g_i = qu.qwen_image_to_patches(Image.fromarray(img), min_pixels=qu.QWEN_VL_UTILS_MIN_PIXELS,
                                           max_pixels=qu.QWEN_VL_UTILS_MAX_PIXELS)
    grids = [g_v, g_s, g_i]
    spg = [qu.second_per_grid(2), qu.second_per_grid(2), 1.0]
    unit = cfg.spatial_merge_size ** 2
    ids, ans = [], []
    tok = FakeTokenizer()
    for k in range(len(paths)):
        t, gh, gw = grids[k]
        vis = cfg.image_token_id if k == 2 else cfg.video_token_id
        for text in texts:
            ids.append(torch.tensor(qu.build_prompt_ids(tok, qu.default_question_template.format(text), t * gh * gw // unit, vis)))
            ans.append(tok.encode("Yes")[0])
    of = [k for k in range(len(paths)) for _ in texts]
    px = torch.cat([rows_v, rows_s, rows_i])
    o32 = qo.qwen25vl_score(sd, ocfg, px, grids, ids, ans, of, mode="fp32", second_per_grid_ts=spg)
    o16 = qo.qwen25vl_score(sd, ocfg, px, grids, ids, ans, of, mode="bf16", second_per_grid_ts=spg)
    gap = float((torch.log(o16) - torch.log(o32)).abs().max())
    err = float((torch.log(got) - torch.log(o32)).abs().max())
    print(f"\n[plugin video mix] grids {grids} engine {got.tolist()} oracle {o32.tolist()} |dlogp| {err:.3e} (oracle bf16-vs-fp32 {gap:.3e})")
    assert got.shape == (6,)
    assert err <= 2.0 * gap + 2e-2
    probs, traces = model.forward_with_trace(pair_paths, pair_texts)
    assert torch.equal(probs, got) and len(traces) == 6


def test_qwen25vl_7b_video_matches_reference_bf16_on_this_gpu(dev):
    """Qwen2.5-VL-7B dims on the realistic video shape: 40 frames of 640x360 sampled at 8 fps -> grid (20, 20, 36), 3600 video tokens,
    S ~ 3.65k; one video x 3 texts in one engine prefill (KV-prefix sharing) against the real HF model in bf16 with sdpa, sample by
    sample, with the video's second_per_grid_ts. The language-model attention runs at this length nowhere else in the suite."""
    import hf_reference as hf
    from t2v_metrics_b200 import _lib
    from t2v_metrics_b200.config import Qwen25VLConfig
    from t2v_metrics_b200.engine import QwenVLEngine, qwen_video_preprocess_u8
    cfg = qo.Qwen25VLConfig.qwen25_vl_7b()
    B, answer = 3, 9454
    rng = np.random.default_rng(11)
    base = rng.integers(0, 256, (40, 45, 80, 3), dtype=np.uint8)
    frames = torch.from_numpy(np.repeat(np.repeat(base, 8, 1), 8, 2).copy())            # 40 x 360 x 640
    mx = int(qu.video_max_pixels(40))
    px, grids = qwen_video_preprocess_u8([frames], [_lib.VQA_RESAMPLE_TORCHVISION], dev, [qu.VIDEO_MIN_PIXELS], [mx])
    assert grids == [(20, 20, 36)]
    spg = qu.second_per_grid(2)
    g = torch.Generator().manual_seed(3)
    n_tok = 20 * 20 * 36 // 4
    prompts = []
    for b in range(B):
        pre = torch.randint(0, 9000, (14,), generator=g).tolist()
        post = torch.randint(0, 9000, (20 + 7 * b,), generator=g).tolist()
        prompts.append(pre + [cfg.video_token_id] * n_tok + post)
    sd = qo.make_synthetic_state_dict(cfg, seed=0, gen_device=dev)
    model = hf.build_hf_qwen(cfg, sd, dtype=torch.bfloat16, device=dev, attn="sdpa")
    pcpu = px.cpu()
    score = lambda: hf.hf_qwen_reference_scores(model, cfg, pcpu.repeat(B, 1), grids * B, prompts, [answer] * B, video=True,
                                                second_per_grid_ts=[spg] * B, return_hidden=True)
    _, hid = score()
    row = hf.calibrate_rows(hid, model.lm_head.weight, answer, torch.tensor([-1.5, 0.0, 1.5]))
    model.lm_head.weight.data[answer] = row.to(dev)
    sd["lm_head.weight"][answer] = row.to(sd["lm_head.weight"].device)
    ref, _ = score()
    del model
    gc.collect()
    torch.cuda.empty_cache()
    fields = {f.name for f in dataclasses.fields(Qwen25VLConfig)}
    eng = QwenVLEngine(Qwen25VLConfig(**{k: v for k, v in dataclasses.asdict(cfg).items() if k in fields}), dev)
    eng.load_state_dict(sd)
    p = eng.score_prompts(px, grids, prompts, [answer] * B, image_of_sample=[0] * B, second_per_grid_ts=[spg]).cpu()
    err = float((p - ref).abs().max())
    print(f"\n[qwen-7b video S={max(map(len, prompts))}] engine {p.tolist()}  HF bf16 sdpa GPU {ref.tolist()}  max|dp| {err:.3e}")
    del sd, eng
    gc.collect()
    torch.cuda.empty_cache()
    assert float(ref.min()) > 0.08 and float(ref.max()) < 0.92
    assert err <= 1e-3, (p, ref)
