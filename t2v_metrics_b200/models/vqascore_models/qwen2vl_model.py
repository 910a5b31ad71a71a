"""Qwen2.5-VL VQAScore plugin backed by the B200 engine (images, video files and 4-D .npy frame stacks).

Same plugin contract as the reference's `Qwen2VLModel` (t2v_metrics/models/vqascore_models/qwen2vl_model.py:93-301): class
attributes, `forward(images, texts, question_template, answer_template, temperature) -> CPU fp32 Tensor[n]` with
score = softmax(last-position logits / temperature)[first answer token]. The reference loops over samples and calls
`generate(max_new_tokens=1)`; here the whole batch is ONE prefill in libvqa_b200.so and identical images or videos are encoded once.
Videos follow qwen_vl_utils.fetch_video (frame sampling and sizing restated in qwen_utils); files are decoded by cv2 on the host
instead of decord, and every frame's resize, normalisation and temporal pairing runs in one device kernel.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import torch

from ...config import QWEN25VL_MODELS as _TABLE, Qwen25VLConfig
from ...constants import HF_CACHE_DIR
from .qwen_utils import (QWEN_VL_UTILS_MAX_PIXELS, QWEN_VL_UTILS_MIN_PIXELS, REFERENCE_VIDEO_FPS, REFERENCE_VIDEO_MAX_PIXELS,
                         VIDEO_EXTENSIONS, VIDEO_MIN_PIXELS, build_prompt_ids, decode_video_cv2,
                         default_answer_template, default_question_template, qwen_image_to_patches, second_per_grid,
                         video_max_pixels)
from .vqa_model import VQAScoreModel

QWEN2_VL_MODELS: Dict[str, dict] = {name: dict(model=dict(path=spec["weights"]), config=spec["config"]) for name, spec in _TABLE.items()}




def _generation_config_penalty(checkpoint_path: str) -> float:
    """repetition_penalty of the generation_config.json stored beside the checkpoint (what `from_pretrained` would attach to
    `model.generation_config` in the reference, qwen2vl_model.py:116-130); 1.0 when there is none."""
    from ...checkpoint import generation_config_value
    return float(generation_config_value(checkpoint_path, "repetition_penalty", 1.0) or 1.0)


class Qwen2VLModel(VQAScoreModel):
    video_mode = "direct"
    allows_image = True
    supports_trace = True

    def __init__(self, model_name="qwen2.5-vl-7b", device="cuda", cache_dir=HF_CACHE_DIR, tokenizer=None,
                 state_dict: Optional[Dict[str, torch.Tensor]] = None, config: Optional[Qwen25VLConfig] = None,
                 checkpoint: Optional[str] = None, repetition_penalty: Optional[float] = None,
                 min_pixels: int = QWEN_VL_UTILS_MIN_PIXELS, max_pixels: int = QWEN_VL_UTILS_MAX_PIXELS, **kwargs):
        assert model_name in QWEN2_VL_MODELS
        self.min_pixels, self.max_pixels = int(min_pixels), int(max_pixels)
        # The reference's scores come out of `generate(..., output_scores=True)`, i.e. AFTER the logits processors the checkpoint's
        # generation_config.json configures (SURVEY F8; Qwen2.5-VL-Instruct ships repetition_penalty 1.05). None = read it from the
        # generation_config.json next to `checkpoint` when there is one, else 1.0 (off).
        self.repetition_penalty = repetition_penalty
        self._tokenizer_override, self._state_dict, self._config_override, self._checkpoint = tokenizer, state_dict, config, checkpoint
        super().__init__(model_name=model_name, device=device, cache_dir=cache_dir)

    def load_model(self):
        from ...engine import QwenVLEngine
        spec = QWEN2_VL_MODELS[self.model_name]
        self.cfg: Qwen25VLConfig = self._config_override or spec["config"]()
        if self._tokenizer_override is not None:
            self.tokenizer = self._tokenizer_override
        else:
            from transformers import AutoTokenizer
            self.tokenizer = AutoTokenizer.from_pretrained(spec["model"]["path"], cache_dir=self.cache_dir)
        from ...checkpoint import load_state_dict, normalise_qwen_keys
        sd = self._state_dict
        if sd is None:
            # a local file or a downloaded repository directory (index json + shards), as `from_pretrained(path)` takes (qwen2vl_model.py:116-130)
            sd = load_state_dict(self._checkpoint or spec["model"]["path"])
        sd = normalise_qwen_keys(sd)      # published checkpoints use `visual.*` / `model.layers.*`; transformers renames them while loading
        if self.repetition_penalty is None:
            self.repetition_penalty = _generation_config_penalty(self._checkpoint or spec["model"]["path"])
        dev = torch.device(self.device if self.device != "cuda" else "cuda:0")
        self.engine = QwenVLEngine(self.cfg, dev)
        self.engine.load_state_dict(sd)
        self._state_dict = None

    def load_images(self, image: List[str], fps=None):
        """-> (patches fp32 [sum rows, 1176] on the device, [(t, gh, gw), ...], second_per_grid_ts per input, is_video per input), in
        the order of `image`. Any mix of image files, 3-D .npy images, 4-D .npy frame stacks and video files (.mp4/.avi/.mov/.mkv);
        `fps` applies to video files: None -> the model table's 8.0, a number, or "dynamic" (qwen_vl_utils' default FPS)."""
        # Host work is decoding only (PIL for images, cv2 for files); smart_resize, the resize (PIL-exact for images and frame stacks,
        # torchvision-exact for decoded files), normalisation, temporal pairing and merge-order patch rows run in one device kernel per
        # kind -- bit-identical to qwen_utils.qwen_image_to_patches / qwen_video_to_patches, the CPU path the reference runs per sample.
        import numpy as np
        from PIL import Image
        from ... import _lib
        from ...engine import qwen_preprocess_u8, qwen_video_preprocess_u8
        fps = REFERENCE_VIDEO_FPS if fps is None else fps
        stills, videos = [], []      # (position, uint8 tensor); videos: (position, frames, policy, min_pixels, max_pixels)
        for i, p in enumerate(image):
            low = p.lower()
            if low.endswith(VIDEO_EXTENSIONS):
                frames, _, _ = decode_video_cv2(p, fps)
                videos.append((i, torch.from_numpy(frames), _lib.VQA_RESAMPLE_TORCHVISION, VIDEO_MIN_PIXELS,
                               int(video_max_pixels(len(frames), REFERENCE_VIDEO_MAX_PIXELS))))
            elif low.endswith(".npy"):
                # the reference's Qwen path takes the array as RGB, no channel flip (qwen2vl_model.py:146-158)
                arr = np.load(p)
                if arr.ndim == 4:         # a frame stack: a list of PIL frames through fetch_video's list branch
                    arr = np.ascontiguousarray(arr.astype("uint8")[..., :3])
                    if arr.shape[-1] != 3 or arr.shape[0] == 0:
                        raise ValueError(f"Unexpected shape for NumPy array in {p}")
                    videos.append((i, torch.from_numpy(arr), _lib.VQA_RESAMPLE_PIL, self.min_pixels, self.max_pixels))
                    continue
                if arr.ndim != 3:
                    raise ValueError(f"Unexpected shape for NumPy array in {p}")
                arr = np.asarray(Image.fromarray(arr.astype("uint8"), "RGB"), dtype=np.uint8)
                stills.append((i, torch.from_numpy(np.ascontiguousarray(arr))))
            else:
                with Image.open(p) as im:
                    stills.append((i, torch.from_numpy(np.ascontiguousarray(np.asarray(im.convert("RGB"), dtype=np.uint8)))))
        dev, cfg = self.engine.device, self.cfg
        parts, order = [], []
        if stills:
            pt, g = qwen_preprocess_u8([t for _, t in stills], dev, cfg.patch_size, cfg.temporal_patch_size, cfg.spatial_merge_size,
                                       min_pixels=self.min_pixels, max_pixels=self.max_pixels)
            parts.append(pt)
            order += [(i, grid, 1.0, False) for (i, _), grid in zip(stills, g)]
        if videos:
            pt, g = qwen_video_preprocess_u8([v[1] for v in videos], [v[2] for v in videos], dev, [v[3] for v in videos],
                                             [v[4] for v in videos], cfg.patch_size, cfg.temporal_patch_size, cfg.spatial_merge_size)
            parts.append(pt)
            # what the reference's processor passes for every video on transformers 5.x (qwen_utils.PROCESSOR_FALLBACK_FPS)
            order += [(v[0], grid, second_per_grid(cfg.temporal_patch_size), True) for v, grid in zip(videos, g)]
        # rows must follow the order of `image`: stills come first, so reorder only when a video precedes an image
        if [o[0] for o in order] != list(range(len(image))):
            rows = [o[1][0] * o[1][1] * o[1][2] for o in order]
            starts = [sum(rows[:k]) for k in range(len(rows))]
            flat = torch.cat(parts)
            by_pos = sorted(range(len(order)), key=lambda k: order[k][0])
            patches = torch.cat([flat[starts[k]:starts[k] + rows[k]] for k in by_pos])
            order = [order[k] for k in by_pos]
        else:
            patches = parts[0] if len(parts) == 1 else torch.cat(parts)
        return patches, [o[1] for o in order], [o[2] for o in order], [o[3] for o in order]

    @torch.no_grad()
    def forward_with_trace(self, images: List[str], texts: List[str], fps=None, question_template: str = default_question_template,
                           answer_template: str = default_answer_template, max_new_tokens: int = 1, temperature: float = 1.0,
                           score_position: str = "end", debug: bool = False, repetition_penalty: Optional[float] = None):
        """Scores plus the per-sample trace dictionaries of the reference's forward_with_trace (qwen2vl_model.py:303-493; schema at
        :469-487): the greedy token, the answer token's probability and the five most probable alternatives. With one generated position
        `score_position` "start" and "end" coincide. The alternatives come from a top-k pass over the last position's logits
        (engine.topk_last) under the same temperature / repetition penalty as the score."""
        assert score_position in ("start", "end"), f"score_position must be 'start' or 'end', got '{score_position}'"
        probs = self.forward(images, texts, fps=fps, question_template=question_template, answer_template=answer_template,
                             max_new_tokens=max_new_tokens, temperature=temperature, debug=False, repetition_penalty=repetition_penalty)
        pen = self.repetition_penalty if repetition_penalty is None else repetition_penalty
        ids, top_p = self.engine.topk_last(5, temperature=temperature, repetition_penalty=pen)
        ids, top_p = ids.cpu().tolist(), top_p.cpu().tolist()
        dec = lambda t: self.tokenizer.decode([t]) if hasattr(self.tokenizer, "decode") else str(t)
        special = {getattr(self.tokenizer, n, None) for n in ("eos_token_id", "bos_token_id", "pad_token_id")} - {None}
        traces = []
        for b, (p, answer_id) in enumerate(zip(probs.tolist(), self._last_answer_ids)):
            generated = ids[b][0]                                   # generate(max_new_tokens=1, do_sample=False) emits the arg-max
            if generated in special:
                # the reference drops a trailing special token and then has nothing left to score (qwen2vl_model.py:395-419)
                raise ValueError("No tokens available to score at the specified position")
            alternatives = [dict(token_id=t, token_text=dec(t), probability=q) for t, q in zip(ids[b], top_p[b])]
            detail = dict(position=0, expected_token_id=answer_id, expected_token_text=dec(answer_id), probability=p, top_alternatives=alternatives)
            traces.append(dict(generated_text=dec(generated), generated_length=1, score_position=score_position, score_start_idx=0,
                               scored_indices=[0], scored_tokens_text=dec(generated), probability=p, token_details=[detail]))
            if debug:
                print(f"sample {b}: generated {dec(generated)!r}; P(answer {dec(answer_id)!r}) = {p:.6f}; top-5 "
                      f"{[(a['token_text'], round(a['probability'], 6)) for a in alternatives]}")
        return probs, traces

    @torch.no_grad()
    def forward(self, images: List[str], texts: List[str], fps=None, question_template: str = default_question_template,
                answer_template: str = default_answer_template, max_new_tokens: int = 1, temperature: float = 1.0,
                debug: bool = False, repetition_penalty: Optional[float] = None) -> torch.Tensor:
        assert len(images) == len(texts), "Number of images/videos and texts must match"
        if max_new_tokens != 1:
            # With max_new_tokens = k > 1 the reference scores answer token i on the logits of generation step len(scores) - n + i, i.e.
            # conditioned on its own GREEDY continuation (qwen2vl_model.py:259-289) -- a decode loop, not the single prefill this engine runs.
            raise NotImplementedError("the B200 engine scores the first generated position only (max_new_tokens=1, the reference default)")
        questions = [question_template.format(t) for t in texts]
        answers = [answer_template.format(t) for t in texts]
        uniq: Dict[str, int] = {}
        index = [uniq.setdefault(p, len(uniq)) for p in images]
        patches, grids, spg, is_video = self.load_images(list(uniq.keys()), fps)
        unit = self.cfg.spatial_merge_size ** 2
        prompts, answer_ids = [], []
        cache = self.__dict__.setdefault("_prompt_cache", {})
        if len(cache) > 65536:
            cache.clear()
        for q, a, img in zip(questions, answers, index):
            t, gh, gw = grids[img]
            token = self.cfg.video_token_id if is_video[img] else self.cfg.image_token_id
            prompts.append(build_prompt_ids(self.tokenizer, q, t * gh * gw // unit, token, cache))
            ids = cache.get(("answer", a))
            if ids is None:
                ids = cache[("answer", a)] = tuple(self.tokenizer.encode(a, add_special_tokens=False))
            if not ids:
                raise ValueError("empty answer")
            # one generated position => the reference truncates a multi-token answer to its first token ("Generated 1 tokens but need n,
            # adjusting", qwen2vl_model.py:259-263) and the geometric mean over one token is that token's probability
            answer_ids.append(ids[0])
        self._last_answer_ids = list(answer_ids)
        probs = self.engine.score_prompts(patches, grids, prompts, answer_ids, image_of_sample=index, temperature=temperature,
                                          repetition_penalty=self.repetition_penalty if repetition_penalty is None else repetition_penalty,
                                          second_per_grid_ts=spg if any(is_video) else None)
        return probs.float().cpu()
