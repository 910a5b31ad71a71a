"""Host-side logic of the drop-in boundary: tokenizer splice, expand2square, preprocessing, registry/API surface, sharding.
CPU only."""
import os
import types

import numpy as np
import pytest
import torch
from PIL import Image

import t2v_metrics_b200 as t2v
from t2v_metrics_b200.models.vqascore_models import mm_utils
from t2v_metrics_b200.models.vqascore_models.clip_t5_model import format_question, CLIP_T5_MODELS, CLIPT5Model
from t2v_metrics_b200.parallel import shard_bounds
from oracle import clipt5_oracle as orc


class FakeTok:
    """Same contract as the generator in tools/make_golden.py: per-word ids + trailing </s> = 1."""
    pad_token_id = 0

    def __call__(self, chunk):
        return types.SimpleNamespace(input_ids=[3 + (sum(map(ord, w)) % 997) for w in chunk.split()] + [1])


def test_golden_vestiges_from_reference(golden_dir):
    """expand2square / t5_tokenizer_image_token outputs recorded by running /root/reference's own mm_utils.py."""
    blob = torch.load(os.path.join(golden_dir, "host_vestiges.pt"), weights_only=False)
    for case in blob["expand2square"]:
        img = Image.fromarray(case["inp"].numpy())
        for fn in (mm_utils.expand2square, orc.expand2square):
            out = np.asarray(fn(img, (122, 116, 104)))
            assert np.array_equal(out, case["out"].numpy())
    for case in blob["t5_tokenizer_image_token"]:
        assert mm_utils.t5_tokenizer_image_token(case["prompt"], FakeTok()) == case["ids"]
        assert orc.t5_tokenizer_image_token(case["prompt"], lambda c: FakeTok()(c).input_ids) == case["ids"]


def test_tokenizer_chunk_cache_is_exact_and_saves_calls():
    """SURVEY 8(f)3: the memo returns exactly what the uncached call returns and tokenises each distinct chunk once."""
    class Counting(FakeTok):
        calls = 0

        def __call__(self, chunk):
            Counting.calls += 1
            return super().__call__(chunk)

    tok, cache = Counting(), {}
    prompts = [f"sys USER: <image>\nDoes this figure show \"{c}\"? ASSISTANT: " for c in ("a dog", "two cats", "a dog", "a dog")]
    plain = [mm_utils.t5_tokenizer_image_token(p, FakeTok()) for p in prompts]
    cached = [mm_utils.t5_tokenizer_image_token(p, tok, chunk_cache=cache) for p in prompts]
    assert cached == plain
    assert Counting.calls == 3            # the shared system chunk + two distinct caption chunks
    from t2v_metrics_b200.models.vqascore_models.qwen_utils import build_prompt_ids

    class QTok:
        calls = 0

        def encode(self, s, add_special_tokens=False):
            QTok.calls += 1
            return [5 + (ord(c) % 89) for c in s]

    qc = {}
    a = [build_prompt_ids(QTok(), q, 4, 600, qc) for q in ("x?", "y?", "x?")]
    b = [build_prompt_ids(QTok(), q, 4, 600) for q in ("x?", "y?", "x?")]
    assert a == b and a[0].count(600) == 4


def test_tokenizer_each_chunk_keeps_its_eos():
    ids = mm_utils.t5_tokenizer_image_token("a <image>\nb", FakeTok())
    assert ids.count(-200) == 1 and ids[ids.index(-200) - 1] == 1 and ids[-1] == 1


def test_prompt_format_matches_reference_constants():
    q = format_question('Does this figure show "a dog"? Please answer yes or no.')
    assert q.startswith("A chat between a curious user") and " USER: <image>\n" in q and q.endswith(" ASSISTANT: ")
    assert q == orc.format_question('Does this figure show "a dog"? Please answer yes or no.')


def test_clip_preprocess_matches_hf_processor():
    from transformers import CLIPImageProcessor
    rng = np.random.RandomState(0)
    proc = CLIPImageProcessor(size={"shortest_edge": 336}, crop_size={"height": 336, "width": 336}, do_resize=True,
                              do_center_crop=True, do_normalize=True, image_mean=list(mm_utils.CLIP_IMAGE_MEAN),
                              image_std=list(mm_utils.CLIP_IMAGE_STD), resample=3, do_convert_rgb=True)
    for (w, h) in [(512, 512), (640, 400), (300, 500)]:
        img = Image.fromarray(rng.randint(0, 256, (h, w, 3), dtype=np.uint8))
        sq = mm_utils.expand2square(img, tuple(int(x * 255) for x in mm_utils.CLIP_IMAGE_MEAN))
        ref = torch.from_numpy(np.asarray(proc.preprocess(sq, return_tensors="np")["pixel_values"][0]))
        got = mm_utils.clip_preprocess(img, 336, pad=True)
        assert got.shape == (3, 336, 336)
        assert float((got - ref).abs().max()) < 2e-2          # PIL vs processor resampling paths, <= 1 grey level
        assert float((got - orc.clip_preprocess(img, 336)).abs().max()) == 0.0


def test_registry_surface_matches_reference():
    assert t2v.list_all_models() == ["clip-flant5-xxl", "clip-flant5-xl", "qwen2.5-vl-7b"]
    assert CLIPT5Model.video_mode == "concat" and CLIPT5Model.allows_image
    assert set(CLIP_T5_MODELS["clip-flant5-xxl"]) >= {"tokenizer", "model"}
    with pytest.raises(NotImplementedError):
        t2v.get_score_model("not-a-model")
    cfg = CLIP_T5_MODELS["clip-flant5-xxl"]["config"]()
    assert (cfg.d_model, cfg.n_heads, cfg.d_ff, cfg.vocab, cfg.num_patches) == (4096, 64, 10240, 32128, 576)


def test_engine_refuses_without_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from t2v_metrics_b200.engine import ClipT5Engine
    from t2v_metrics_b200.config import ClipT5Config
    with pytest.raises(RuntimeError):
        ClipT5Engine(ClipT5Config())


@pytest.mark.parametrize("n,world", [(10000, 8), (7, 8), (64, 1), (65, 2), (0, 4)])
def test_shard_bounds_cover_all_pairs_once(n, world):
    seen = []
    for r in range(world):
        s, e, per = shard_bounds(n, world, r)
        assert 0 <= s <= e <= n and e - s <= per
        seen.extend(range(s, e))
    assert seen == list(range(n))


def test_qwen_patch_layout_matches_hf_processor():
    """a19: smart_resize + patch flattening vs transformers' Qwen2VLImageProcessor (do_resize=False on a pre-sized image, as the
    reference calls it after qwen_vl_utils resized the image: qwen2vl_model.py:208-216)."""
    from transformers.models.qwen2_vl.image_processing_qwen2_vl import Qwen2VLImageProcessor, smart_resize as hf_smart_resize
    from t2v_metrics_b200.models.vqascore_models.qwen_utils import smart_resize, qwen_image_to_patches
    for hw in [(448, 448), (500, 333), (30, 4000), (2000, 3000), (57, 57)]:
        assert smart_resize(*hw) == hf_smart_resize(*hw)
    rng = np.random.RandomState(0)
    proc = Qwen2VLImageProcessor()
    for (h, w) in [(448, 448), (84, 140)]:
        img = Image.fromarray(rng.randint(0, 256, (h, w, 3), dtype=np.uint8))
        ref = proc(images=[img], do_resize=False, return_tensors="pt")
        got, grid = qwen_image_to_patches(img)
        assert list(grid) == ref["image_grid_thw"][0].tolist()
        assert float((got - ref["pixel_values"]).abs().max()) < 1e-5


def test_prompt_constants_equal_the_reference_module(golden_dir):
    """The prompt constants are part of the model's training recipe: compare with the values of the reference's own
    t2v_metrics/constants.py, recorded in golden/reference_constants.json."""
    import json
    from t2v_metrics_b200 import constants as c
    assert c.IMAGE_TOKEN_INDEX == -200 and c.IGNORE_INDEX == -100 and c.DEFAULT_IMAGE_TOKEN == "<image>" and c.CONTEXT_LEN == 2048
    assert c.SYSTEM_MSG.startswith("A chat between a curious user") and c.SYSTEM_MSG.endswith("to the user's questions.")
    with open(os.path.join(golden_dir, "reference_constants.json")) as f:
        ref = json.load(f)
    assert set(ref) == {"HF_CACHE_DIR", "CONTEXT_LEN", "SYSTEM_MSG", "IGNORE_INDEX", "IMAGE_TOKEN_INDEX", "DEFAULT_IMAGE_TOKEN"}
    for k, v in ref.items():
        assert getattr(c, k) == v, k


def test_image_loader_cases(tmp_path):
    """.npy = BGR array reversed to RGB; everything else through PIL, always 3-channel RGB (reference model.py:10-14)."""
    from t2v_metrics_b200.models.model import image_loader
    a = (np.arange(4 * 5 * 3) % 255).astype(np.uint8).reshape(4, 5, 3)
    np.save(tmp_path / "x.npy", a)
    Image.fromarray(a).save(tmp_path / "x.png")
    Image.fromarray(a[:, :, 0]).save(tmp_path / "g.png")
    assert (np.asarray(image_loader(str(tmp_path / "x.npy"))) == a[:, :, ::-1]).all()
    assert (np.asarray(image_loader(str(tmp_path / "x.png"))) == a).all()
    assert np.asarray(image_loader(str(tmp_path / "g.png"))).shape == (4, 5, 3)


def test_checkpoint_directory_shards_and_key_names(tmp_path):
    """mm_utils.py:182-241 / qwen2vl_model.py:110-133 load HF repository directories: index json + shards, on-disk tensor names. The
    loader returns the in-memory HF names the engine converters consume, for either naming."""
    import json
    from safetensors.torch import save_file
    from oracle import qwen25vl_oracle as qo
    from t2v_metrics_b200 import checkpoint as ck
    cfg = qo.Qwen25VLConfig.tiny()
    sd = qo.make_synthetic_state_dict(cfg)
    disk = {}
    for k, v in sd.items():           # the names published Qwen2.5-VL checkpoints carry on disk
        if k.startswith("model.visual."):
            disk[k[len("model."):]] = v
        elif k.startswith("model.language_model."):
            disk["model." + k[len("model.language_model."):]] = v
        else:
            disk[k] = v
    keys = sorted(disk)
    wm = {}
    for i, part in enumerate((keys[: len(keys) // 2], keys[len(keys) // 2:])):
        name = f"model-0000{i + 1}-of-00002.safetensors"
        save_file({k: disk[k].contiguous() for k in part}, str(tmp_path / name))
        wm.update({k: name for k in part})
    (tmp_path / "model.safetensors.index.json").write_text(json.dumps(dict(metadata={}, weight_map=wm)))
    (tmp_path / "generation_config.json").write_text(json.dumps(dict(repetition_penalty=1.05)))
    back = ck.normalise_qwen_keys(ck.load_state_dict(str(tmp_path)))
    assert set(back) == set(sd) and all(torch.equal(back[k], sd[k]) for k in sd)
    assert set(ck.normalise_qwen_keys(sd)) == set(sd)                                  # already in-memory names: unchanged
    assert ck.generation_config_value(str(tmp_path), "repetition_penalty", 1.0) == 1.05
    assert ck.generation_config_value(str(tmp_path / "model-00001-of-00002.safetensors"), "repetition_penalty", 1.0) == 1.05
    with pytest.raises(FileNotFoundError, match="no network"):
        ck.load_state_dict(str(tmp_path / "absent"))
    # CLIP-FlanT5: LLaVA-style nesting, vision tower inside the checkpoint or loaded separately (mm_utils.py:226-227)
    c = orc.ClipT5Config.tiny()
    s = orc.make_synthetic_state_dict(c)
    llava, vis = {}, {}
    for k, v in s.items():
        if k.startswith("vision_tower."):
            vis[k[len("vision_tower."):]] = v
        elif k.startswith("mm_projector."):
            llava["model." + k] = v
        else:
            llava[k] = v
    assert set(ck.normalise_clipt5_keys(llava, vis)) == set(s)
    nested = dict(llava, **{"model.vision_tower.vision_tower." + k: v for k, v in vis.items()})
    assert set(ck.normalise_clipt5_keys(nested)) == set(s)
    with pytest.raises(KeyError, match="vision_tower_checkpoint"):
        ck.normalise_clipt5_keys(llava)


def test_qwen_resize_bounds_follow_qwen_vl_utils_not_the_hf_processor():
    """The reference resizes in qwen_vl_utils.process_vision_info (MIN_PIXELS = 4*28*28, MAX_PIXELS = 16384*28*28) and calls the HF
    processor with do_resize=False (reference qwen2vl_model.py:201-216): the processor's 14*14*4*1280 ceiling must not apply. The
    reference's own images/0.png (1920 x 1280) is above that ceiling."""
    from t2v_metrics_b200.engine import qwen_preprocess_plan
    from t2v_metrics_b200.models.vqascore_models import qwen2vl_model as qm
    from t2v_metrics_b200.models.vqascore_models.qwen_utils import smart_resize
    assert (qm.QWEN_VL_UTILS_MIN_PIXELS, qm.QWEN_VL_UTILS_MAX_PIXELS) == (3136, 12845056)
    ref_like = smart_resize(1280, 1920, 28, qm.QWEN_VL_UTILS_MIN_PIXELS, qm.QWEN_VL_UTILS_MAX_PIXELS)
    assert ref_like == (1288, 1932)                                       # round to multiples of 28, no down-scaling
    hf_default = smart_resize(1280, 1920)                                 # the processor's own bound: scaled down to <= 1 003 520 pixels
    assert hf_default[0] * hf_default[1] <= 14 * 14 * 4 * 1280 < ref_like[0] * ref_like[1]
    assert smart_resize(1024, 1024, 28, qm.QWEN_VL_UTILS_MIN_PIXELS, qm.QWEN_VL_UTILS_MAX_PIXELS) == (1036, 1036)   # ADVICE r1: 1369 tokens, not 1225
    for bounds in ((qm.QWEN_VL_UTILS_MIN_PIXELS, qm.QWEN_VL_UTILS_MAX_PIXELS), (56 * 56, 14 * 14 * 4 * 1280)):
        sizes = [(1280, 1920), (1275, 1920), (1024, 1024), (20, 30), (5000, 4000)]
        grids, _, _ = qwen_preprocess_plan(sizes, min_pixels=bounds[0], max_pixels=bounds[1])   # the C++ plan the device kernel uses
        assert [(g[1] * 14, g[2] * 14) for g in grids] == [smart_resize(h, w, 28, *bounds) for h, w in sizes]
    import inspect
    sig = inspect.signature(qm.Qwen2VLModel.__init__)
    assert sig.parameters["max_pixels"].default == qm.QWEN_VL_UTILS_MAX_PIXELS and sig.parameters["min_pixels"].default == qm.QWEN_VL_UTILS_MIN_PIXELS


def test_plugins_refuse_inputs_the_kernels_cannot_take():
    """ADVICE r1: a caption containing '<image>' adds a second image slot (the splice kernel handles exactly one); Qwen max_new_tokens > 1
    needs the reference's greedy decode loop. Both must fail loudly on the host, before anything is launched."""
    from t2v_metrics_b200.models.vqascore_models import qwen2vl_model as qm
    fake = types.SimpleNamespace(tokenizer=FakeTok(), context_len=2048, cfg=types.SimpleNamespace(vocab=32128))
    q = format_question('Does this figure show "{}"? Please answer yes or no.'.format("a dog"))
    ids, lens, labels = CLIPT5Model._tokenize(fake, [q], ["Yes"])
    assert int((ids == -200).sum()) == 1 and int(lens[0]) == ids.shape[1]
    bad = format_question('Does this figure show "{}"? Please answer yes or no.'.format("a dog <image> and a cat"))
    with pytest.raises(ValueError, match="exactly one"):
        CLIPT5Model._tokenize(fake, [bad], ["Yes"])
    with pytest.raises(ValueError, match="answer"):
        CLIPT5Model._tokenize(fake, [q], ["<image>"])
    with pytest.raises(NotImplementedError, match="max_new_tokens=1"):
        qm.Qwen2VLModel.forward(types.SimpleNamespace(), ["a.png"], ["a dog"], max_new_tokens=2)


def test_small_calls_are_bucketed_for_cuda_graph_replay():
    """Calls with <= cuda_graph_max_pairs pairs pad the id matrix to a multiple of 16 columns (few call shapes -> few captured graphs); the true
    lengths stay in `lens` (the engine masks the padding), and larger calls keep the tight width."""
    fake = types.SimpleNamespace(tokenizer=FakeTok(), context_len=2048, cfg=types.SimpleNamespace(vocab=32128, pad_token_id=0), cuda_graph_max_pairs=4)
    qs = [format_question('Does this figure show "{}"? Please answer yes or no.'.format(t)) for t in ("a dog", "two cats on a mat", "x")]
    ids, lens, labels = CLIPT5Model._tokenize(fake, qs, ["Yes"] * 3)
    assert ids.shape[1] % 16 == 0 and ids.shape[1] - int(lens.max()) < 16
    for i in range(3):
        assert bool((ids[i, int(lens[i]):] == 0).all()) and int((ids[i] == -200).sum()) == 1
    fake.cuda_graph_max_pairs = 2
    ids2, lens2, _ = CLIPT5Model._tokenize(fake, qs, ["Yes"] * 3)
    assert ids2.shape[1] == int(lens2.max()) and torch.equal(lens, lens2) and torch.equal(ids[:, : ids2.shape[1]], ids2)
