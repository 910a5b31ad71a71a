"""Qwen2.5-VL video scoring, timed end to end from uint8 frames, at qwen2.5-vl-7b width with synthetic weights (one process, one GPU).

  (a) config-5 shape: 8 in-memory frame stacks of 16 frames of 224x224 (grid 8x16x16, 512 video tokens), one text each. Times what
      Qwen2VLModel.forward does after loading: the device pre-processing (PIL-exact resize, pairing, patch rows), the host index
      building, the prefill and the copy of the scores to the host. Comparable to `bench.py --video`'s e2e, which starts from the
      processor's fp32 patch rows instead of uint8 frames.
  (b) a realistic file: 5 s of 640x360 at 24 fps written to a temporary .mp4, sampled at 8 fps (40 frames, grid 20x20x36, 3600 video
      tokens, S ~ 3.65k), scored against 8 texts. Host decode (cv2) is reported apart from the device part (pre-processing, indices,
      prefill with the video's prefix shared by the 8 prompts, D2H).

Each case prints one JSON line, with the GPU's name and power limit read in the same run:
    python tools/bench_qwen_video.py --steps 20 --warmup 3 [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def gpu_info(index: int) -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i", str(index)],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return dict(gpu=out[0], power_limit_w=float(out[1]))
    except Exception:
        return dict(gpu=torch.cuda.get_device_name(index), power_limit_w=None)


def timed(fn, steps: int, warmup: int, dev) -> list:
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize(dev)
    ms = []
    for _ in range(steps):
        t0 = time.perf_counter()
        fn()                              # ends with a device -> host copy of the scores, i.e. a synchronise
        ms.append((time.perf_counter() - t0) * 1e3)
    return ms


def summary(ms):
    ms = sorted(ms)
    return dict(median_ms=round(ms[len(ms) // 2], 3), min_ms=round(ms[0], 3), max_ms=round(ms[-1], 3))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_qwen_video.py measures on a GPU; none is visible")
    from t2v_metrics_b200 import _lib, qwen_host
    from t2v_metrics_b200.config import QWEN25VL_MODELS
    from t2v_metrics_b200.engine import QwenVLEngine, qwen_video_preprocess_u8
    from t2v_metrics_b200.models.vqascore_models import qwen_utils as qu
    from t2v_metrics_b200.synthetic import synthetic_qwen_engine_weights

    dev = torch.device("cuda:0")
    info = gpu_info(0)
    cfg = QWEN25VL_MODELS["qwen2.5-vl-7b"]["config"]()
    eng = QwenVLEngine(cfg, dev)
    eng.bind_engine_tensors(synthetic_qwen_engine_weights(cfg, dev, seed=0))
    rng = np.random.default_rng(0)
    g = torch.Generator().manual_seed(1)
    unit = cfg.spatial_merge_size ** 2
    spg = qu.second_per_grid(cfg.temporal_patch_size)
    lines = []

    def prompt(n_vis, text_len):
        pre = torch.randint(0, 9000, (14,), generator=g).tolist()
        return pre + [cfg.video_token_id] * n_vis + torch.randint(0, 9000, (text_len,), generator=g).tolist()

    def score(videos, policies, mins, maxs, prompts, image_of_sample):
        px, grids = qwen_video_preprocess_u8(videos, policies, dev, mins, maxs, cfg.patch_size, cfg.temporal_patch_size,
                                             cfg.spatial_merge_size)
        p = eng.score_prompts(px, grids, prompts, [9454] * len(prompts), image_of_sample=image_of_sample,
                              second_per_grid_ts=[spg] * len(grids))
        return p.cpu(), grids

    # ---- (a) config-5 shape from in-memory frame stacks
    B = 8
    stacks = [torch.from_numpy(rng.integers(0, 256, (16, 224, 224, 3), dtype=np.uint8)).pin_memory() for _ in range(B)]
    prompts_a = [prompt(8 * 16 * 16 // unit, 50) for _ in range(B)]
    args_a = (stacks, [_lib.VQA_RESAMPLE_PIL] * B, [qu.QWEN_VL_UTILS_MIN_PIXELS] * B, [qu.QWEN_VL_UTILS_MAX_PIXELS] * B, prompts_a,
              list(range(B)))
    _, grids_a = score(*args_a)
    ms = timed(lambda: score(*args_a), args.steps, args.warmup, dev)
    s = summary(ms)
    lines.append(dict(case="a_config5_frame_stacks", model="qwen2.5-vl-7b", weights="synthetic", batch=B, frames=16, frame_hw=[224, 224],
                      grid_thw=list(grids_a[0]), seq_len=max(map(len, prompts_a)), **s,
                      pairs_per_s=round(B / (s["median_ms"] / 1e3), 2), steps=args.steps, warmup=args.warmup, **info))

    # ---- (b) realistic file: 5 s of 640x360 at 24 fps, fps 8, one video x 8 texts
    import cv2
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "clip.mp4")
        wr = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"mp4v"), 24.0, (640, 360))
        if not wr.isOpened():
            raise SystemExit("this OpenCV build cannot write mp4v")
        base = rng.integers(0, 256, (120, 45, 80, 3), dtype=np.uint8)
        for f in np.repeat(np.repeat(base, 8, 1), 8, 2):
            wr.write(f)
        wr.release()
        dec = []
        for _ in range(max(args.steps // 4, 3)):
            t0 = time.perf_counter()
            frames, _, idx = qu.decode_video_cv2(path, qu.REFERENCE_VIDEO_FPS)
            dec.append((time.perf_counter() - t0) * 1e3)
    n = len(frames)
    mx = int(qu.video_max_pixels(n))
    vid = torch.from_numpy(frames).pin_memory()
    rh, rw = qu.video_frame_size(*frames.shape[1:3], n)
    n_vis = (n // 2) * (rh // 14) * (rw // 14) // unit
    prompts_b = [prompt(n_vis, 12 + 3 * k) for k in range(8)]
    prompts_b = [prompts_b[0][:14 + n_vis] + p[14 + n_vis:] for p in prompts_b]     # the same chat prefix: one video, 8 questions
    args_b = ([vid], [_lib.VQA_RESAMPLE_TORCHVISION], [qu.VIDEO_MIN_PIXELS], [mx], prompts_b, [0] * 8)
    _, grids_b = score(*args_b)
    ms = timed(lambda: score(*args_b), args.steps, args.warmup, dev)
    s = summary(ms)
    lines.append(dict(case="b_file_640x360_5s_fps8_x8_texts", model="qwen2.5-vl-7b", weights="synthetic", texts=8, frames=n,
                      frame_hw=[360, 640], resized_hw=[rh, rw], grid_thw=list(grids_b[0]), seq_len=max(map(len, prompts_b)),
                      host_decode_ms=summary(dec)["median_ms"], device_ms=s["median_ms"], device_min_ms=s["min_ms"],
                      device_max_ms=s["max_ms"], steps=args.steps, warmup=args.warmup, **info))
    for line in lines:
        print(json.dumps(line), flush=True)
    if args.out:
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
