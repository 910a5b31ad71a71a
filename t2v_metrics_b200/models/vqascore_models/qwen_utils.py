"""Host-side image / prompt preparation of the Qwen2.5-VL path.

* `smart_resize` + `qwen_image_to_patches`: what `qwen_vl_utils.process_vision_info` (PIL resize to multiples of 28) and
  `Qwen2VLImageProcessor._preprocess` with do_resize=False (transformers/models/qwen2_vl/image_processing_qwen2_vl.py:62-87,
  :191-220) do to one still image: rescale, CLIP-normalise, duplicate the frame along the temporal axis, cut 14x14 patches and
  emit them in 2x2 merge-block order as rows of 3*2*14*14 = 1176 values.
* `build_prompt_ids`: the chat template the reference applies (qwen2vl_model.py:197-200) with the image (or video) pad expanded to
  one token per merged patch group (processing_qwen2_5_vl.py:119-137).
* Videos: the frame sampling and sizing of `qwen_vl_utils.vision_process.fetch_video` (`smart_nframes`, `sample_frame_indices`,
  `video_max_pixels`, `video_frame_size`), the two resizes it applies (`pil_resize_frames` for frame lists, `torchvision_resize_u8` for
  decoded files), the cv2 decoder that stands in for decord (`decode_video_cv2`) and `qwen_video_to_patches`, what
  `Qwen2VLVideoProcessor` with do_resize=False does to the resized frames.
"""
from __future__ import annotations

import math
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch
from PIL import Image

OPENAI_CLIP_MEAN = (0.48145466, 0.4578275, 0.40821073)
OPENAI_CLIP_STD = (0.26862954, 0.26130258, 0.27577711)

default_question_template = 'Does this figure show "{}"? Please answer Yes or No.'   # qwen2vl_model.py:173
default_answer_template = "Yes"                                                        # qwen2vl_model.py:174

# Pixel bounds of the resize the reference applies to still images BEFORE the HF processor: `process_vision_info`
# (qwen_vl_utils.vision_process.fetch_image) calls smart_resize(h, w, factor=28, min_pixels=MIN_PIXELS, max_pixels=MAX_PIXELS) with
# MIN_PIXELS = 4 * 28 * 28 and MAX_PIXELS = 16384 * 28 * 28, and the processor then runs with do_resize=False (reference
# qwen2vl_model.py:201-216), so the processor's own 14*14*4*1280 ceiling never applies. qwen_vl_utils is an unpinned dependency that
# is not installed here: the two values are restated from its source and exposed as constructor arguments (`min_pixels=`,
# `max_pixels=`) for other versions. Frames of a 4-D .npy stack go through the same fetch_image, so they use the same bounds.
QWEN_VL_UTILS_MIN_PIXELS = 4 * 28 * 28
QWEN_VL_UTILS_MAX_PIXELS = 16384 * 28 * 28

# Video constants of qwen_vl_utils.vision_process, restated from memory of that package's source: UNVERIFIED against an installed
# copy (none can be installed here). Each names the module-level constant or function it comes from.
VIDEO_MIN_PIXELS = 128 * 28 * 28                    # VIDEO_MIN_PIXELS: floor of a video frame's smart_resize
VIDEO_MAX_PIXELS = 768 * 28 * 28                    # VIDEO_MAX_PIXELS: per-frame ceiling before the total-budget split
VIDEO_TOTAL_PIXELS = int(128000 * 28 * 28 * 0.9)    # VIDEO_TOTAL_PIXELS (its default; the package lets an env variable override it)
FRAME_FACTOR = 2                                    # FRAME_FACTOR: frame counts are multiples of 2 (one temporal patch)
FPS = 2.0                                           # FPS: sampling rate of fetch_video when the caller gives none
FPS_MIN_FRAMES = 4                                  # FPS_MIN_FRAMES: smart_nframes lower clamp
FPS_MAX_FRAMES = 768                                # FPS_MAX_FRAMES: smart_nframes upper clamp
FRAME_LIST_SAMPLE_FPS = 2.0                         # fetch_video, list branch: `process_info.pop("fps", 2.0)` with no fps given
# What the reference plugin itself passes with a video file ({"video": path, "max_pixels": 360*420, "fps": fps}, reference
# qwen2vl_model.py:141-146) and the fps of its model table (`fps` absent -> 8.0, :138).
REFERENCE_VIDEO_MAX_PIXELS = 360 * 420
REFERENCE_VIDEO_FPS = 8.0
VIDEO_EXTENSIONS = (".mp4", ".avi", ".mov", ".mkv")

CHAT_PREFIX = "<|im_start|>system\nYou are a helpful assistant.<|im_end|>\n<|im_start|>user\n<|vision_start|>"
CHAT_SUFFIX = "<|vision_end|>{question}<|im_end|>\n<|im_start|>assistant\n"


def smart_resize(height: int, width: int, factor: int = 28, min_pixels: int = 56 * 56, max_pixels: int = 14 * 14 * 4 * 1280) -> Tuple[int, int]:
    """Both sides divisible by `factor`, pixel count within [min_pixels, max_pixels], aspect ratio kept as closely as possible."""
    if max(height, width) / min(height, width) > 200:
        raise ValueError("absolute aspect ratio must be smaller than 200")
    h_bar = round(height / factor) * factor
    w_bar = round(width / factor) * factor
    if h_bar * w_bar > max_pixels:
        beta = math.sqrt((height * width) / max_pixels)
        h_bar = max(factor, math.floor(height / beta / factor) * factor)
        w_bar = max(factor, math.floor(width / beta / factor) * factor)
    elif h_bar * w_bar < min_pixels:
        beta = math.sqrt(min_pixels / (height * width))
        h_bar = math.ceil(height * beta / factor) * factor
        w_bar = math.ceil(width * beta / factor) * factor
    return h_bar, w_bar


def qwen_image_to_patches(img: Image.Image, patch_size: int = 14, temporal_patch_size: int = 2, merge_size: int = 2,
                          min_pixels: int = 56 * 56, max_pixels: int = 14 * 14 * 4 * 1280):
    """One RGB image -> (patches fp32 [gh*gw, 3*temporal*ps*ps], (1, gh, gw))."""
    img = img.convert("RGB")
    w, h = img.size
    rh, rw = smart_resize(h, w, patch_size * merge_size, min_pixels, max_pixels)
    if (rw, rh) != (w, h):
        img = img.resize((rw, rh), resample=Image.BICUBIC)
    x = torch.from_numpy(np.asarray(img, dtype=np.float32)).permute(2, 0, 1) / 255.0
    x = (x - torch.tensor(OPENAI_CLIP_MEAN)[:, None, None]) / torch.tensor(OPENAI_CLIP_STD)[:, None, None]
    x = x[None].repeat(temporal_patch_size, 1, 1, 1)                      # still image: the frame is duplicated
    gh, gw = rh // patch_size, rw // patch_size
    x = x.view(1, temporal_patch_size, 3, gh // merge_size, merge_size, patch_size, gw // merge_size, merge_size, patch_size)
    x = x.permute(0, 3, 6, 4, 7, 2, 1, 5, 8)                             # (t, h/m, w/m, m, m, c, tp, ps, ps)
    return x.reshape(gh * gw, 3 * temporal_patch_size * patch_size * patch_size).contiguous(), (1, gh, gw)


def build_prompt_ids(tokenizer, question: str, n_image_tokens: int, image_token_id: int, cache: Optional[dict] = None) -> List[int]:
    """`cache` (SURVEY 8(f)3): exact memo string -> ids; the chat prefix is constant and M x N scoring repeats each question M times.
    `image_token_id` is the vision pad of the run: <|image_pad|> for images, <|video_pad|> for videos (same chat template)."""
    def enc(s: str):
        if cache is None:
            return list(tokenizer.encode(s, add_special_tokens=False))
        ids = cache.get(s)
        if ids is None:
            ids = cache[s] = tuple(tokenizer.encode(s, add_special_tokens=False))
        return list(ids)
    return enc(CHAT_PREFIX) + [image_token_id] * n_image_tokens + enc(CHAT_SUFFIX.format(question=question))


# ------------------------------------------------------------------------------------------------ video (qwen_vl_utils.vision_process)
def round_by_factor(number: float, factor: int) -> int:
    return round(number / factor) * factor


def ceil_by_factor(number: float, factor: int) -> int:
    return math.ceil(number / factor) * factor


def floor_by_factor(number: float, factor: int) -> int:
    return math.floor(number / factor) * factor


def smart_nframes(total_frames: int, video_fps: float, fps: float = FPS) -> int:
    """vision_process.smart_nframes for an element with `fps` (no `nframes`): total / video_fps * fps, clamped to
    [ceil2(FPS_MIN_FRAMES), floor2(min(FPS_MAX_FRAMES, total))] and to total, then floored to a multiple of FRAME_FACTOR."""
    min_frames = ceil_by_factor(FPS_MIN_FRAMES, FRAME_FACTOR)
    max_frames = floor_by_factor(min(FPS_MAX_FRAMES, total_frames), FRAME_FACTOR)
    nframes = total_frames / video_fps * fps
    nframes = min(min(max(nframes, min_frames), max_frames), total_frames)
    nframes = floor_by_factor(nframes, FRAME_FACTOR)
    if not (FRAME_FACTOR <= nframes <= total_frames):
        raise ValueError(f"nframes should in interval [{FRAME_FACTOR}, {total_frames}], but got {nframes}.")
    return int(nframes)


def sample_frame_indices(total_frames: int, nframes: int) -> List[int]:
    """The frames fetch_video's readers keep: torch.linspace(0, total - 1, nframes).round() (fp32 linspace, round-half-even)."""
    return torch.linspace(0, total_frames - 1, nframes).round().long().tolist()


def video_sample_fps(nframes: int, total_frames: int, video_fps: float) -> float:
    """The rate the readers report for the sampled frames: nframes / total * video_fps."""
    return nframes / max(total_frames, 1e-6) * video_fps


def video_max_pixels(nframes: int, max_pixels: Optional[int] = REFERENCE_VIDEO_MAX_PIXELS) -> float:
    """fetch_video's per-frame pixel budget: min(max_pixels, max(min(VIDEO_MAX_PIXELS, VIDEO_TOTAL_PIXELS / nframes * FRAME_FACTOR),
    int(VIDEO_MIN_PIXELS * 1.05))); `max_pixels` is the element's own value (None = not given)."""
    budget = max(min(VIDEO_MAX_PIXELS, VIDEO_TOTAL_PIXELS / nframes * FRAME_FACTOR), int(VIDEO_MIN_PIXELS * 1.05))
    return budget if max_pixels is None else min(max_pixels, budget)


def video_frame_size(height: int, width: int, nframes: int, max_pixels: Optional[int] = REFERENCE_VIDEO_MAX_PIXELS) -> Tuple[int, int]:
    """(resized_height, resized_width) of a decoded video's frames: smart_resize(h, w, 28, VIDEO_MIN_PIXELS, video_max_pixels)."""
    return smart_resize(height, width, 28, VIDEO_MIN_PIXELS, video_max_pixels(nframes, max_pixels))


# transformers 5.5 Qwen2_5_VLProcessor.__call__ sets second_per_grid_ts = temporal_patch_size / VideoMetadata.sampled_fps. The reference
# hands over already-sampled frames and the reader's rate as an `fps` keyword, which the 5.x video processor only uses to SAMPLE
# frames (off with pre-sampled input); with no metadata, sampled_fps falls back to 24 (transformers/video_utils.py). So on the
# transformers this project targets, every video gets 2 / 24 whatever its sampling rate (older transformers used 2 / fps).
PROCESSOR_FALLBACK_FPS = 24.0


def second_per_grid(temporal_patch_size: int = 2, video_fps: Optional[float] = None) -> float:
    """second_per_grid_ts of one video as the installed processor computes it: temporal_patch_size / the metadata's fps, which is
    PROCESSOR_FALLBACK_FPS when, as in the reference, no metadata is passed."""
    return temporal_patch_size / (video_fps or PROCESSOR_FALLBACK_FPS)


def decode_video_cv2(path: str, fps=REFERENCE_VIDEO_FPS, max_frames: Optional[int] = None):
    """Decode a video file the way fetch_video reads it, with cv2 in place of decord: count the frames by reading them, take the rate
    from CAP_PROP_FPS, sample smart_nframes of them (fps="dynamic" -> the package default FPS) and keep only those, BGR -> RGB.
    Returns (frames uint8 [n, h, w, 3], sample_fps, indices). cv2 and decord may decode the same file to slightly different frames (and
    count a damaged file differently); that is a known deviation from the reference, not a parity claim."""
    try:
        import cv2
    except ImportError as e:
        raise ImportError("decoding video files needs OpenCV (pip install opencv-python-headless); 4-D .npy frame stacks do not") from e
    fps = FPS if fps == "dynamic" else float(fps)
    cap = cv2.VideoCapture(path)
    if not cap.isOpened():
        raise ValueError(f"cannot open video file {path}")
    try:
        video_fps = float(cap.get(cv2.CAP_PROP_FPS))
        total = 0
        while cap.grab():
            total += 1
    finally:
        cap.release()
    if total == 0 or not video_fps > 0:
        raise ValueError(f"no decodable frames (or no frame rate) in {path}")
    nframes = smart_nframes(total, video_fps, fps)
    idx = sample_frame_indices(total, nframes)
    want: dict = {}
    for k, i in enumerate(idx):
        want.setdefault(i, []).append(k)
    frames: List[Optional[np.ndarray]] = [None] * nframes
    cap = cv2.VideoCapture(path)
    try:
        i = 0
        while i <= idx[-1] and cap.grab():
            if i in want:
                ok, bgr = cap.retrieve()
                if not ok:
                    raise ValueError(f"cannot decode frame {i} of {path}")
                rgb = cv2.cvtColor(bgr, cv2.COLOR_BGR2RGB)
                for k in want[i]:
                    frames[k] = rgb
            i += 1
    finally:
        cap.release()
    if any(f is None for f in frames):
        raise ValueError(f"{path} ended before frame {idx[-1]}")
    return np.stack(frames), video_sample_fps(nframes, total, video_fps), idx


def torchvision_resize_u8(frames: torch.Tensor, height: int, width: int) -> torch.Tensor:
    """uint8 [T, h, w, 3] -> uint8 [T, height, width, 3], what fetch_video's
    `transforms.functional.resize(video, [h, w], BICUBIC, antialias=True)` returns for a uint8 tensor: an fp32 antialiased bicubic
    (F.interpolate), clamp to [0, 255], round half to even. (fetch_video then calls .float(), which changes no value.)"""
    x = frames.permute(0, 3, 1, 2).float()
    if (height, width) != tuple(x.shape[-2:]):
        x = torch.nn.functional.interpolate(x, size=(height, width), mode="bicubic", antialias=True)
    return x.clamp(0, 255).round().to(torch.uint8).permute(0, 2, 3, 1).contiguous()


def pil_resize_frames(frames: np.ndarray, min_pixels: int = QWEN_VL_UTILS_MIN_PIXELS,
                      max_pixels: int = QWEN_VL_UTILS_MAX_PIXELS) -> np.ndarray:
    """A frame list through fetch_video's list branch: every frame through fetch_image (smart_resize with the image bounds, PIL
    BICUBIC), then the count rounded up to a multiple of FRAME_FACTOR by repeating the last frame. uint8 [T, h, w, 3] -> [T', rh, rw, 3]."""
    out = []
    for f in frames:
        img = Image.fromarray(np.asarray(f, dtype=np.uint8), "RGB")
        rh, rw = smart_resize(img.height, img.width, 28, min_pixels, max_pixels)
        out.append(np.asarray(img.resize((rw, rh), resample=Image.BICUBIC) if (rh, rw) != (img.height, img.width) else img))
    out += [out[-1]] * (ceil_by_factor(len(out), FRAME_FACTOR) - len(out))
    return np.stack(out)


def qwen_video_to_patches(frames, patch_size: int = 14, temporal_patch_size: int = 2, merge_size: int = 2):
    """Resized frames (uint8 [T, h, w, 3], h and w multiples of patch_size * merge_size) -> (patches fp32
    [T/tp * gh * gw, 3*tp*ps*ps], (T/tp, gh, gw)): Qwen2VLVideoProcessor with do_resize=False -- rescale, CLIP-normalise,
    consecutive frames paired into one temporal patch (a count that is not a multiple of tp repeats the last frame), rows in
    merge-block order. Same fp32 arithmetic as qwen_image_to_patches."""
    x = torch.as_tensor(np.asarray(frames, dtype=np.uint8)).permute(0, 3, 1, 2).float() / 255.0
    x = (x - torch.tensor(OPENAI_CLIP_MEAN)[:, None, None]) / torch.tensor(OPENAI_CLIP_STD)[:, None, None]
    if x.shape[0] % temporal_patch_size:
        x = torch.cat([x, x[-1:].repeat(temporal_patch_size - x.shape[0] % temporal_patch_size, 1, 1, 1)])
    T, _, h, w = x.shape
    gt, gh, gw = T // temporal_patch_size, h // patch_size, w // patch_size
    x = x.view(gt, temporal_patch_size, 3, gh // merge_size, merge_size, patch_size, gw // merge_size, merge_size, patch_size)
    x = x.permute(0, 3, 6, 4, 7, 2, 1, 5, 8)                             # (t, h/m, w/m, m, m, c, tp, ps, ps)
    return x.reshape(gt * gh * gw, 3 * temporal_patch_size * patch_size * patch_size).contiguous(), (gt, gh, gw)
