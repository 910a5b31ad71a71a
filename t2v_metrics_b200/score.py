"""Score orchestration above the plugin boundary -- same call surface as the reference's t2v_metrics/score.py
(`Score.forward` :47-113 -> [M, N] tensor on `device`; `Score.batch_forward` :115-156 -> [samples, visuals, texts]).

Differences, all above the drop-in boundary and result-preserving:
  * `forward` hands ALL M x N pairs to the plugin in one call (chunked by `max_pairs`); the plugin encodes each distinct
    image once. The reference loops `self.model.forward([image] * N, texts)` per image (score.py:104-106).
  * `batch_forward` scores a whole DataLoader batch per (visual, text) slot, as v3.0 did, instead of one pair at a time
    (v3.1 score.py:143-153).
  * video paths go to plugins with `video_mode == "direct"` (Qwen2.5-VL), which sample, resize and encode the frames themselves.
    The cv2 frame-concatenation path of `video_mode == "concat"` plugins (reference score.py:72-98) is not built and raises.
"""
from typing import List, Optional, TypedDict, Union

import torch
import torch.nn as nn

from .constants import HF_CACHE_DIR

VIDEO_EXTENSIONS = {'.mp4', '.avi', '.mov', '.mkv'}


class ImageTextDict(TypedDict):
    images: List[str]
    texts: List[str]


class Score(nn.Module):
    def __init__(self, model: str, device: str = 'cuda', cache_dir: str = HF_CACHE_DIR, **kwargs):
        super().__init__()
        assert model in self.list_all_models()
        self.device = device
        self.model = self.prepare_scoremodel(model, device, cache_dir, **kwargs)
        self.model_name = model
        self.max_pairs = 64
        # Opt-in for one process per GPU (torchrun) when EVERY rank calls forward() with the SAME images and texts: the IMAGES are split over
        # the ranks, so that every image's vision features are computed on one rank only, and the [m, n] score rows are all-gathered
        # (SURVEY 8e). Off (default): every rank scores what it is given, like the reference -- ranks may then hold different data.
        self.shard_over_images = False

    def prepare_scoremodel(self, model: str, device: str, cache_dir: str, **kwargs):
        raise NotImplementedError("Subclasses must implement prepare_scoremodel")

    def list_all_models(self) -> List[str]:
        raise NotImplementedError("Subclasses must implement list_all_models")

    def forward(self, images: Optional[Union[str, List[str]]] = None, texts: Optional[Union[str, List[str]]] = None,
                num_frames: Optional[int] = 8, **kwargs) -> torch.Tensor:
        """m images x n texts -> [m, n] tensor of scores on self.device."""
        if isinstance(images, str):
            images = [images]
        if isinstance(texts, str):
            texts = [texts]
        if any(isinstance(img, str) and img[-4:].lower() in VIDEO_EXTENSIONS for img in images) and \
                getattr(self.model, "video_mode", None) != "direct":
            raise NotImplementedError("video inputs (frame extraction + concat, reference score.py:72-98) are outside the "
                                      "B200 engine's hot-path scope for this model; pass image files or use a direct-video model")
        m, n = len(images), len(texts)
        import torch.distributed as dist
        world = dist.get_world_size() if (self.shard_over_images and dist.is_available() and dist.is_initialized()) else 1
        if world > 1:
            from .parallel import shard_bounds
            start, end, per = shard_bounds(m, world, dist.get_rank())
        else:
            start, end, per = 0, m, m
        pair_images = [img for img in images[start:end] for _ in range(n)]
        pair_texts = [t for _ in range(end - start) for t in texts]
        out = [torch.zeros(0)]
        for s in range(0, len(pair_images), self.max_pairs):
            out.append(self.model.forward(pair_images[s:s + self.max_pairs], pair_texts[s:s + self.max_pairs], **kwargs).float().cpu())
        local = torch.cat(out)
        if world > 1:
            # equal-sized shards of `per` images (the last ranks may hold fewer or none: zero rows, trimmed after the gather)
            dev = torch.device(self.device) if dist.get_backend() == "nccl" else torch.device("cpu")
            padded = torch.zeros(per * n, dtype=torch.float32, device=dev)
            padded[: local.numel()] = local.to(dev)
            gathered = torch.empty(world * per * n, dtype=torch.float32, device=dev)
            dist.all_gather_into_tensor(gathered, padded)
            local = gathered[: m * n]
        return local.view(m, n).to(self.device)

    def batch_forward(self, dataset: List[ImageTextDict], batch_size: int = 16, num_frames: int = 4, **kwargs) -> torch.Tensor:
        """[num_samples, num_visuals, num_texts] scores for a dataset of {'images': [...], 'texts': [...]} items, or, for models with
        `video_mode == "direct"`, of {'videos': [...], 'texts': [...]} items, scored exactly like images (the plugin takes the paths).
        The reference's own video branch calls `self.forward(videos=...)`, a keyword its forward does not accept; here video datasets
        go through the same per-slot plugin calls as images instead."""
        from torch.utils.data import DataLoader
        num_samples = len(dataset)
        key = 'images'
        if "videos" in dataset[0]:
            if getattr(self.model, "video_mode", None) != "direct":
                raise NotImplementedError("video datasets need a model with video_mode 'direct'; the concat path is not built")
            key = 'videos'
        num_visuals = len(dataset[0][key])
        num_texts = len(dataset[0]['texts'])
        scores = torch.zeros(num_samples, num_visuals, num_texts).to(self.device)
        dataloader = DataLoader(dataset, batch_size=batch_size, shuffle=False)
        counter = 0
        for batch_idx, batch in enumerate(dataloader):
            cur = len(batch[key][0])
            assert len(batch[key]) == num_visuals and len(batch['texts']) == num_texts
            for vis_idx in range(num_visuals):
                for text_idx in range(num_texts):
                    scores[counter:counter + cur, vis_idx, text_idx] = self.model.forward(
                        list(batch[key][vis_idx]), list(batch['texts'][text_idx]), **kwargs).to(self.device)
            counter += cur
        return scores
