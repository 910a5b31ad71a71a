"""Tensor-level entry to the B200 engine: PyTorch tensors in, PyTorch tensors out, everything in between is
libvqa_b200.so (hand-written sm_100a kernels) reached through ctypes. PyTorch only supplies device memory and the
current CUDA stream.

`ClipT5Engine.score_tensors` is what `bench.py` and the plugin (`models/clip_t5_model.py`) call; it replaces the
`self.model(input_ids, images=..., labels=...)` + CrossEntropy loop of the reference's v3.0 CLIPT5Model.forward.
"""
from __future__ import annotations

import collections
import ctypes as C
from typing import Dict, Optional, Sequence

import torch

from . import _lib
from .config import ClipT5Config

IMAGE_TOKEN_INDEX = -200  # t2v_metrics/constants.py:7
IGNORE_INDEX = -100       # t2v_metrics/constants.py:6


def _ptr(t: Optional[torch.Tensor]):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _stream_ptr(device) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _check(rc: int, handle=None, what: str = ""):
    if rc != 0:
        raise RuntimeError(f"libvqa_b200 {what} failed (status {rc}): {_lib.last_error(handle)}")


def fold_norm_gain(weight: torch.Tensor, gamma: torch.Tensor) -> torch.Tensor:
    """W . diag(gamma) in fp32, rounded to bf16 once: the weight the fused-norm GEMMs use (their epilogue supplies rsqrt(mean(x^2) + eps))."""
    return (weight.float() * gamma.float()[None, :]).to(torch.bfloat16).contiguous()


def convert_state_dict(sd: Dict[str, torch.Tensor], cfg: ClipT5Config, device, fuse_norms: bool = False) -> Dict[str, torch.Tensor]:
    """HF-named CLIP-FlanT5 weights (CLIPVisionModel under `vision_tower.`, `mm_projector.*`,
    T5ForConditionalGeneration names) -> the engine's fused bf16 layout:
      * q/k/v projections concatenated row-wise ([3*inner, d]) so one GEMM produces the packed QKV buffer;
      * wi_0 / wi_1 concatenated ([2*d_ff, d]) for the gated-GELU epilogue; cross-attention k/v concatenated;
      * the Conv2d patch embedding flattened to [D, 3*ps*ps] and zero-padded along K to a multiple of 64.
    Mirrors `model.to(device, dtype=torch.bfloat16)` (mm_utils.py:228)."""
    out: Dict[str, torch.Tensor] = {}

    def put(name, t):
        out[name] = t.detach().to(device=device, dtype=torch.bfloat16).contiguous()

    v = "vision_tower.vision_model."
    D = cfg.vit_hidden
    k_real = 3 * cfg.patch_size * cfg.patch_size
    kpad = (k_real + 63) // 64 * 64
    pw = sd[v + "embeddings.patch_embedding.weight"].reshape(D, k_real)
    pw_pad = torch.zeros(D, kpad, dtype=pw.dtype, device=pw.device)
    pw_pad[:, :k_real] = pw
    put("vit.patch_embed.weight", pw_pad)
    put("vit.class_embedding", sd[v + "embeddings.class_embedding"])
    put("vit.position_embedding", sd[v + "embeddings.position_embedding.weight"])
    put("vit.pre_ln.weight", sd[v + "pre_layrnorm.weight"])
    put("vit.pre_ln.bias", sd[v + "pre_layrnorm.bias"])
    for l in range(cfg.vit_layers - 1):
        p, q = v + f"encoder.layers.{l}.", f"vit.layers.{l}."
        put(q + "ln1.weight", sd[p + "layer_norm1.weight"]); put(q + "ln1.bias", sd[p + "layer_norm1.bias"])
        put(q + "ln2.weight", sd[p + "layer_norm2.weight"]); put(q + "ln2.bias", sd[p + "layer_norm2.bias"])
        put(q + "qkv.weight", torch.cat([sd[p + f"self_attn.{n}_proj.weight"] for n in "qkv"], dim=0))
        put(q + "qkv.bias", torch.cat([sd[p + f"self_attn.{n}_proj.bias"] for n in "qkv"], dim=0))
        put(q + "out.weight", sd[p + "self_attn.out_proj.weight"]); put(q + "out.bias", sd[p + "self_attn.out_proj.bias"])
        put(q + "fc1.weight", sd[p + "mlp.fc1.weight"]); put(q + "fc1.bias", sd[p + "mlp.fc1.bias"])
        put(q + "fc2.weight", sd[p + "mlp.fc2.weight"]); put(q + "fc2.bias", sd[p + "mlp.fc2.bias"])
    for i in (0, 2):
        put(f"proj.{i}.weight", sd[f"mm_projector.{i}.weight"]); put(f"proj.{i}.bias", sd[f"mm_projector.{i}.bias"])
    put("t5.shared", sd["shared.weight"])
    put("t5.lm_head", sd["lm_head.weight"])  # untied from `shared` for FlanT5 (SURVEY F6)
    put("t5.enc.rel_bias", sd["encoder.block.0.layer.0.SelfAttention.relative_attention_bias.weight"])
    put("t5.dec.rel_bias", sd["decoder.block.0.layer.0.SelfAttention.relative_attention_bias.weight"])
    put("t5.enc.final_ln", sd["encoder.final_layer_norm.weight"])
    put("t5.dec.final_ln", sd["decoder.final_layer_norm.weight"])
    for l in range(cfg.enc_layers):
        p, q = f"encoder.block.{l}.layer.", f"t5.enc.{l}."
        a = p + "0.SelfAttention."
        put(q + "ln0", sd[p + "0.layer_norm.weight"])
        put(q + "qkv", torch.cat([sd[a + f"{n}.weight"] for n in "qkv"], dim=0))
        put(q + "o", sd[a + "o.weight"])
        put(q + "ln1", sd[p + "1.layer_norm.weight"])
        put(q + "wi", torch.cat([sd[p + "1.DenseReluDense.wi_0.weight"], sd[p + "1.DenseReluDense.wi_1.weight"]], dim=0))
        put(q + "wo", sd[p + "1.DenseReluDense.wo.weight"])
        if fuse_norms:
            out[q + "qkv_g"] = fold_norm_gain(out[q + "qkv"], out[q + "ln0"])
            out[q + "wi_g"] = fold_norm_gain(out[q + "wi"], out[q + "ln1"])
    for l in range(cfg.dec_layers):
        p, q = f"decoder.block.{l}.layer.", f"t5.dec.{l}."
        a, c = p + "0.SelfAttention.", p + "1.EncDecAttention."
        put(q + "ln0", sd[p + "0.layer_norm.weight"])
        put(q + "qkv", torch.cat([sd[a + f"{n}.weight"] for n in "qkv"], dim=0))
        put(q + "o", sd[a + "o.weight"])
        put(q + "ln1", sd[p + "1.layer_norm.weight"])
        put(q + "cq", sd[c + "q.weight"])
        put(q + "ckv", torch.cat([sd[c + "k.weight"], sd[c + "v.weight"]], dim=0))
        put(q + "ckT", sd[c + "k.weight"].t())   # Wk^T for the absorbed cross-attention
        put(q + "co", sd[c + "o.weight"])
        put(q + "ln2", sd[p + "2.layer_norm.weight"])
        put(q + "wi", torch.cat([sd[p + "2.DenseReluDense.wi_0.weight"], sd[p + "2.DenseReluDense.wi_1.weight"]], dim=0))
        put(q + "wo", sd[p + "2.DenseReluDense.wo.weight"])
    return out


class ClipT5Engine:
    """One engine = one model replica on one GPU (one process per GPU; SURVEY section 8e)."""

    def __init__(self, cfg: ClipT5Config, device="cuda:0", emulate_bf16_rounding: bool = True,
                 cross_attention_mode: str = "absorbed", round_attention_scores: bool = False, fuse_norms: bool = False):
        """round_attention_scores: form the bf16 score tensors of the reference's eager attention before the softmax (off: fp32 scores --
        closer to the exact result, and measured no closer to the bf16 reference, DESIGN.md section 4). fuse_norms: fold the encoder's
        T5LayerNorms into the GEMMs around them (no normalised copy of the residual stream; a different, equally valid rounding point)."""
        if not torch.cuda.is_available():
            raise RuntimeError("ClipT5Engine needs a CUDA device (sm_100a); there is no CPU path")
        self.lib = _lib.load()
        self.cfg = cfg
        self.device = torch.device(device)
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        c = _lib.VqaClipT5Config(
            image_size=cfg.image_size, patch_size=cfg.patch_size, vit_hidden=cfg.vit_hidden, vit_heads=cfg.vit_heads,
            vit_mlp=cfg.vit_mlp, vit_layers_run=cfg.vit_layers - 1, vit_ln_eps=cfg.vit_ln_eps, d_model=cfg.d_model,
            n_heads=cfg.n_heads, d_ff=cfg.d_ff, enc_layers=cfg.enc_layers, dec_layers=cfg.dec_layers, vocab=cfg.vocab,
            rel_buckets=cfg.rel_buckets, rel_max_distance=cfg.rel_max_distance, t5_ln_eps=cfg.t5_ln_eps,
            image_token_id=IMAGE_TOKEN_INDEX, pad_token_id=cfg.pad_token_id, decoder_start_id=cfg.decoder_start_id,
            emulate_bf16_rounding=(1 if emulate_bf16_rounding else 0) | (2 if round_attention_scores else 0) | (4 if fuse_norms else 0),
            cross_attention_mode={"absorbed": 0, "reference": 1}[cross_attention_mode])
        self.fuse_norms = bool(fuse_norms)
        if cfg.d_kv != 64:
            raise ValueError("the engine's attention kernels are specialised for d_kv == 64")
        self._h = C.c_void_p()
        with torch.cuda.device(idx):
            _check(self.lib.vqa_create_clipt5(C.byref(c), idx, C.byref(self._h)), None, "vqa_create_clipt5")
        self._weights: Dict[str, torch.Tensor] = {}
        self._workspace: Optional[torch.Tensor] = None
        self._graphs: Dict[tuple, tuple] = {}      # CUDA graphs of whole forwards, keyed by the call's shapes (score_tensors_graphed)

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            self.lib.vqa_destroy(h)
            self._h = C.c_void_p()

    # ---- weights
    def bind_engine_tensors(self, tensors: Dict[str, torch.Tensor]):
        if getattr(self, "fuse_norms", False) and "t5.enc.0.qkv" in tensors and "t5.enc.0.qkv_g" not in tensors:
            tensors = dict(tensors)       # engine-layout weights without the folded copies (synthetic / shared dicts): derive them
            for l in range(self.cfg.enc_layers):
                q = f"t5.enc.{l}."
                tensors[q + "qkv_g"] = fold_norm_gain(tensors[q + "qkv"], tensors[q + "ln0"])
                tensors[q + "wi_g"] = fold_norm_gain(tensors[q + "wi"], tensors[q + "ln1"])
        arr = (_lib.VqaTensor * len(tensors))()
        keep = []
        for i, (name, t) in enumerate(tensors.items()):
            assert t.is_cuda and t.dtype == torch.bfloat16 and t.is_contiguous(), name
            nb = name.encode()
            keep.append(nb)
            arr[i].name = nb
            arr[i].data = t.data_ptr()
            for d in range(4):
                arr[i].shape[d] = t.shape[d] if d < t.dim() else 1
            arr[i].ndim = t.dim()
            arr[i].dtype = _lib.VQA_DTYPE_BF16
        _check(self.lib.vqa_bind_weights(self._h, arr, len(tensors)), self._h, "vqa_bind_weights")
        self._weights.update(tensors)  # keep the borrowed memory alive
        _check(self.lib.vqa_finalize_weights(self._h), self._h, "vqa_finalize_weights")

    def load_state_dict(self, sd: Dict[str, torch.Tensor]):
        self.bind_engine_tensors(convert_state_dict(sd, self.cfg, self.device, fuse_norms=self.fuse_norms))

    # ---- forward
    def workspace_bytes(self, batch: int, n_images: int, text_len: int, label_len: int) -> int:
        return int(self.lib.vqa_clipt5_workspace_bytes(self._h, batch, n_images, text_len, label_len))

    def score_tensors(self, pixel_values: torch.Tensor, input_ids: torch.Tensor, text_lens: torch.Tensor,
                      labels: torch.Tensor, image_index: Optional[torch.Tensor] = None,
                      out: Optional[torch.Tensor] = None, return_logprobs: bool = False):
        """pixel_values [NI,3,H,W] fp32/bf16 cuda; input_ids [B,L] int32 (-200 = image slot); text_lens [B] int32;
        labels [B,T] int32 (-100 = ignore); image_index [B] int32 or None. Returns scores [B] fp32 on the device
        (enqueued on the current stream; no synchronisation)."""
        dev = self.device
        assert pixel_values.is_cuda and pixel_values.dim() == 4 and pixel_values.is_contiguous()
        assert pixel_values.dtype in (torch.float32, torch.bfloat16)
        for t in (input_ids, text_lens, labels):
            assert t.is_cuda and t.dtype == torch.int32 and t.is_contiguous()
        B, L = input_ids.shape
        T = labels.shape[1]
        NI = pixel_values.shape[0]
        if image_index is not None:
            assert image_index.is_cuda and image_index.dtype == torch.int32 and image_index.shape == (B,)
        need = self.workspace_bytes(B, NI, L, T)
        if self._workspace is None or self._workspace.numel() < need:
            self._graphs.clear()              # captured graphs point into the old workspace
            self._workspace = None
            self._workspace = torch.empty(need, dtype=torch.uint8, device=dev)
        if out is None:
            out = torch.empty(B, dtype=torch.float32, device=dev)
        logp = torch.zeros(B, T, dtype=torch.float32, device=dev) if return_logprobs else None   # ignored (-100) positions stay 0
        pdt = _lib.VQA_DTYPE_F32 if pixel_values.dtype == torch.float32 else _lib.VQA_DTYPE_BF16
        with torch.cuda.device(dev):      # the library launches on the CURRENT device: make it the engine's (a process may drive several GPUs)
            rc = self.lib.vqa_clipt5_score(self._h, _ptr(pixel_values), pdt, NI, _ptr(image_index), _ptr(input_ids),
                                           _ptr(text_lens), _ptr(labels), B, L, T, _ptr(out), _ptr(logp),
                                           _ptr(self._workspace), self._workspace.numel(), _stream_ptr(dev))
        _check(rc, self._h, "vqa_clipt5_score")
        return (out, logp) if return_logprobs else out

    MAX_GRAPHS = 16

    def score_tensors_graphed(self, pixel_values: torch.Tensor, input_ids: torch.Tensor, text_lens: torch.Tensor, labels: torch.Tensor,
                              image_index: Optional[torch.Tensor] = None) -> torch.Tensor:
        """score_tensors replayed from a CUDA graph captured once per call shape (SURVEY 7 step 6): the forward is ~700 launches whose
        host-side cost (launch + argument marshalling) is the floor of small-batch calls such as the M x N API with a handful of pairs.
        Inputs are copied into the graph's static buffers; the returned scores tensor is the graph's output buffer (valid until the next
        replay of the same shape)."""
        key = (tuple(pixel_values.shape), pixel_values.dtype, tuple(input_ids.shape), int(labels.shape[1]), image_index is not None)
        entry = self._graphs.get(key)
        if entry is None:
            static = [t.clone() if t is not None else None for t in (pixel_values, input_ids, text_lens, labels, image_index)]
            self.score_tensors(static[0], static[1], static[2], static[3], image_index=static[4])      # sizes the workspace, sets kernel attributes
            torch.cuda.synchronize(self.device)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                out = self.score_tensors(static[0], static[1], static[2], static[3], image_index=static[4])
            entry = self._graphs[key] = (graph, static, out)
            while len(self._graphs) > self.MAX_GRAPHS:          # oldest shape first (dict order = insertion order)
                self._graphs.pop(next(iter(self._graphs)))
        graph, static, out = entry
        for dst, src in zip(static, (pixel_values, input_ids, text_lens, labels, image_index)):
            if dst is not None:
                dst.copy_(src, non_blocking=True)
        graph.replay()
        return out

    def score_host(self, pixel_values: torch.Tensor, input_ids: torch.Tensor, text_lens: torch.Tensor,
                   labels: torch.Tensor, image_index: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Host tensors in, host tensor out: H2D copies of this step's inputs (use pinned memory for async copies),
        one engine call, D2H of the scores. This is the end-to-end call bench.py's `e2e` times."""
        dev = self.device
        d = [t.to(dev, non_blocking=True) if t is not None else None
             for t in (pixel_values, input_ids, text_lens, labels, image_index)]
        scores = self.score_tensors(d[0], d[1], d[2], d[3], image_index=d[4])
        return scores.cpu()

    def score_images_u8(self, images_u8, input_ids: torch.Tensor, text_lens: torch.Tensor, labels: torch.Tensor,
                        image_index: Optional[torch.Tensor] = None, pad: bool = True) -> torch.Tensor:
        """End to end from DECODED images: uint8 HWC host (pinned) or device tensors -> device pre-processing kernel -> scores on
        the host. The reference does the resize + normalise per image on the CPU (a4 in SURVEY 8a) before its forward."""
        dev = self.device
        pixels = clip_preprocess_u8(images_u8, self.cfg.image_size, dev, pad=pad)
        d = [t.to(dev, non_blocking=True) if t is not None else None for t in (input_ids, text_lens, labels, image_index)]
        return self.score_tensors(pixels, d[0], d[1], d[2], image_index=d[3]).cpu()

    def last_launch_count(self) -> int:
        return int(self.lib.vqa_last_launch_count(self._h))

    def debug_tensors(self, batch: int, n_images: int, text_len: int, label_len: int) -> Dict[str, torch.Tensor]:
        """Views into the workspace of the LAST call with these sizes (synchronise first): encoder / decoder outputs after their
        final norms, projector output, residual streams. Parity investigations only."""
        off = (C.c_size_t * 6)()
        _check(self.lib.vqa_clipt5_debug_layout(self._h, batch, n_images, text_len, label_len, off, 6), self._h, "vqa_clipt5_debug_layout")
        cfg = self.cfg
        S = text_len - 1 + cfg.num_patches
        ws = self._workspace

        def view(o, rows, cols):
            return ws[o:o + rows * cols * 2].view(torch.bfloat16).view(rows, cols)
        return dict(enc_out=view(off[0], batch * S, cfg.d_model).view(batch, S, cfg.d_model),
                    dec_out=view(off[1], batch * label_len, cfg.d_model).view(batch, label_len, cfg.d_model),
                    proj=view(off[2], n_images * (cfg.num_patches + 1), cfg.d_model).view(n_images, cfg.num_patches + 1, cfg.d_model),
                    vit_hidden=ws[off[5]:off[5] + n_images * (cfg.num_patches + 1) * cfg.vit_hidden * 4].view(torch.float32)
                    .view(n_images, cfg.num_patches + 1, cfg.vit_hidden))

    def set_profile(self, enable: bool):
        _check(self.lib.vqa_set_profile(self._h, 1 if enable else 0), self._h, "vqa_set_profile")

    def read_profile(self):
        """After torch.cuda.synchronize(): {category: (device_ms, algorithmic_flops, scopes, algorithmic_bytes)} of the last call."""
        ms = (C.c_float * 4)()
        fl = (C.c_double * 4)()
        by = (C.c_double * 4)()
        sc = (C.c_int64 * 4)()
        _check(self.lib.vqa_profile_read(self._h, ms, fl, by, sc), self._h, "vqa_profile_read")
        names = ("gemm", "attention", "norm", "other")
        return {n: (float(ms[i]), float(fl[i]), int(sc[i]), float(by[i])) for i, n in enumerate(names)}


# ------------------------------------------------------------------------------------------------ single-kernel ops
class ops:
    """Kernel-level calls through the same C ABI (used by tests and bench.py's roofline probe)."""

    EPI = dict(store=0, quick_gelu=1, gelu=2, gated_gelu=3, relu=5)

    @staticmethod
    def gemm(a: torch.Tensor, w: torch.Tensor, bias=None, residual=None, epilogue="store", variant=0, out=None,
             gate_up_offset=0):
        lib = _lib.load()
        M, K = a.shape
        n_rows = w.shape[0]
        epi = ops.EPI[epilogue]
        n_out = n_rows // 2 if epi == 3 else n_rows
        if out is None:
            out = torch.empty(M, n_out, dtype=torch.bfloat16, device=a.device)
        rc = lib.vqa_op_gemm_bf16(_ptr(a), a.stride(0), _ptr(w), w.stride(0), n_rows, _ptr(out), out.stride(0), M, n_rows,
                                  K, _ptr(bias), _ptr(residual), residual.stride(0) if residual is not None else 0, epi,
                                  gate_up_offset if epi == 3 else 0, variant, _stream_ptr(a.device))
        _check(rc, None, "vqa_op_gemm_bf16")
        return out

    @staticmethod
    def gemm_normfuse(a: torch.Tensor, w: torch.Tensor, residual=None, epilogue="store", gate_up_offset=0, ssq_in=None, ssq_out=None,
                      norm_dim: int = 0, eps: float = 1e-6, out=None):
        """GEMM with the fused-RMSNorm hooks (see include/vqa_b200.h). ssq_in / ssq_out: fp32 [M, stride] cuda, stride % 4 == 0.
        Returns (C, number of ssq_out slots written)."""
        lib = _lib.load()
        M, K = a.shape
        n_rows = w.shape[0]
        epi = ops.EPI[epilogue]
        n_out = n_rows // 2 if epi == 3 else n_rows
        if out is None:
            out = torch.empty(M, n_out, dtype=torch.bfloat16, device=a.device)
        buf = ssq_in if ssq_in is not None else ssq_out
        parts = C.c_int32(0)
        rc = lib.vqa_op_gemm_bf16_normfuse(_ptr(a), a.stride(0), _ptr(w), w.stride(0), n_rows, _ptr(out), out.stride(0), M, n_rows, K,
                                           _ptr(residual), residual.stride(0) if residual is not None else 0, epi,
                                           gate_up_offset if epi == 3 else 0, _ptr(ssq_in), _ptr(ssq_out), buf.shape[1], norm_dim or K, float(eps),
                                           C.byref(parts), _stream_ptr(a.device))
        _check(rc, None, "vqa_op_gemm_bf16_normfuse")
        return out, int(parts.value)

    @staticmethod
    def lmhead_logprob(h: torch.Tensor, w: torch.Tensor, labels: torch.Tensor):
        lib = _lib.load()
        M, K = h.shape
        N = w.shape[0]
        ntiles = (N + 127) // 128
        scratch = torch.empty(4 * M * ntiles + M, dtype=torch.float32, device=h.device)
        out = torch.empty(M, dtype=torch.float32, device=h.device)
        rc = lib.vqa_op_lmhead_logprob(_ptr(h), h.stride(0), _ptr(w), w.stride(0), M, N, K, _ptr(labels), _ptr(out),
                                       _ptr(scratch), _stream_ptr(h.device))
        _check(rc, None, "vqa_op_lmhead_logprob")
        return out

    @staticmethod
    def attention(qkv: torch.Tensor, B: int, S: int, H: int, seq_lens=None, bias_table=None, scale=1.0,
                  bias_const_from: int = 0, round_scores: bool = False):
        """bias_const_from > 0 promises that bias_table[h] is constant for |key - query| >= bias_const_from on either side (T5:
        relative_attention_max_distance); 0 makes no assumption. round_scores: form the reference's bf16 score tensors before the softmax."""
        lib = _lib.load()
        out = torch.empty(B * S, H * 64, dtype=torch.bfloat16, device=qkv.device)
        rc = lib.vqa_op_attention_d64(_ptr(qkv), _ptr(out), B, S, H, _ptr(seq_lens), _ptr(bias_table), float(scale),
                                      int(bias_const_from), 1 if round_scores else 0, _stream_ptr(qkv.device))
        _check(rc, None, "vqa_op_attention_d64")
        return out

    @staticmethod
    def norm(x: torch.Tensor, gamma: torch.Tensor, beta=None, eps=1e-6):
        lib = _lib.load()
        y = torch.empty_like(x)
        rc = lib.vqa_op_norm(_ptr(x), _ptr(gamma), _ptr(beta), _ptr(y), x.shape[0], x.shape[1], float(eps),
                             _stream_ptr(x.device))
        _check(rc, None, "vqa_op_norm")
        return y


# ------------------------------------------------------------------------------------------------ image pre-processing
class _PinnedRing:
    """A few pinned host buffers handed to the library as `host_staging`, each guarded by a CUDA event recorded after the call that
    used it, so a buffer is never rewritten before the stream has consumed it (keeps the pre-processing call fully asynchronous)."""

    def __init__(self, slots: int = 4):
        self.bufs = [None] * slots
        self.events = [None] * slots
        self.i = 0

    def acquire(self, nbytes: int) -> torch.Tensor:
        self.i = (self.i + 1) % len(self.bufs)
        if self.events[self.i] is not None:
            self.events[self.i].synchronize()
        if self.bufs[self.i] is None or self.bufs[self.i].numel() < nbytes:
            self.bufs[self.i] = torch.empty(max(nbytes, 1 << 16), dtype=torch.uint8, pin_memory=True)
        return self.bufs[self.i]

    def release(self, device):
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(device))
        self.events[self.i] = ev


_staging_rings: Dict[int, _PinnedRing] = {}


def _staging(device: torch.device) -> _PinnedRing:
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if idx not in _staging_rings:
        _staging_rings[idx] = _PinnedRing()
    return _staging_rings[idx]


CLIP_MEAN = (0.48145466, 0.4578275, 0.40821073)
CLIP_STD = (0.26862954, 0.26130258, 0.27577711)


def clip_preprocess_u8(images: Sequence[torch.Tensor], out_size: int, device, pad: bool = True, mean=CLIP_MEAN, std=CLIP_STD,
                       background=None, out_dtype: torch.dtype = torch.float32, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Decoded images (uint8 HWC RGB tensors, each [h, w, 3], on the host or on `device`) -> CLIP input [n, 3, S, S] on the device,
    by ONE kernel launch of libvqa_b200.so: expand2square (reference mm_utils.py:128-139, background = int(mean * 255)) + PIL-exact
    bicubic resize + centre crop + /255 + normalise. Host images are packed into one pinned buffer and copied once (a 512x512 image
    is 0.79 MB as uint8 against 1.35 MB as the fp32 336x336 tensor the CPU path ships). Enqueued on the current stream."""
    lib = _lib.load()
    dev = torch.device(device)
    n = len(images)
    assert n > 0
    hs, ws, offs, total = [], [], [], 0
    for im in images:
        assert im.dtype == torch.uint8 and im.dim() == 3 and im.shape[2] == 3, "images must be uint8 [h, w, 3]"
        hs.append(int(im.shape[0])); ws.append(int(im.shape[1])); offs.append(total)
        total += int(im.numel())
    if isinstance(images, torch.Tensor):      # one packed [n, h, w, 3] batch of equal-size images: no staging copy
        src = images.contiguous().view(-1)
        src = src if src.is_cuda else src.to(dev, non_blocking=True)
    elif all(im.is_cuda for im in images):
        src = images[0].contiguous().view(-1) if n == 1 else torch.cat([im.contiguous().view(-1) for im in images])
    else:
        stage = torch.empty(total, dtype=torch.uint8, pin_memory=True)
        for im, o in zip(images, offs):
            stage[o:o + im.numel()] = im.contiguous().view(-1)
        src = stage.to(dev, non_blocking=True)
    H = (C.c_int32 * n)(*hs)
    W = (C.c_int32 * n)(*ws)
    O = (C.c_int64 * n)(*offs)
    need = int(lib.vqa_clip_preprocess_workspace_bytes(H, W, n, out_size, 1 if pad else 0))
    if need == 0:
        raise RuntimeError(f"vqa_clip_preprocess_workspace_bytes: {_lib.last_error(None)}")
    wsb = torch.empty(need, dtype=torch.uint8, device=dev)
    if out is None:
        out = torch.empty(n, 3, out_size, out_size, dtype=out_dtype, device=dev)
    assert out.is_cuda and out.is_contiguous() and out.shape == (n, 3, out_size, out_size) and out.dtype in (torch.float32, torch.bfloat16)
    bg = background if background is not None else tuple(int(x * 255) for x in mean)
    ring = _staging(dev)
    hs = ring.acquire(need)
    with torch.cuda.device(dev):
        rc = lib.vqa_clip_preprocess(_ptr(src), O, H, W, n, out_size, 1 if pad else 0, (C.c_uint8 * 3)(*bg), (C.c_float * 3)(*mean),
                                     (C.c_float * 3)(*std), _ptr(out), _lib.VQA_DTYPE_F32 if out.dtype == torch.float32 else _lib.VQA_DTYPE_BF16,
                                     _ptr(wsb), need, hs.data_ptr(), _stream_ptr(dev))
    ring.release(dev)
    _check(rc, None, "vqa_clip_preprocess")
    # src / wsb stay referenced by the caching allocator's stream ordering: both were allocated on the current stream
    return out


def qwen_preprocess_plan(sizes_hw: Sequence[Sequence[int]], patch: int = 14, merge: int = 2, min_pixels: int = 56 * 56,
                         max_pixels: int = 14 * 14 * 4 * 1280):
    """Host-only geometry of the Qwen pre-processing (smart_resize): -> ([(1, gh, gw), ...], total patch rows, workspace bytes)."""
    lib = _lib.load()
    n = len(sizes_hw)
    H = (C.c_int32 * n)(*[int(s[0]) for s in sizes_hw])
    W = (C.c_int32 * n)(*[int(s[1]) for s in sizes_hw])
    grid = (C.c_int32 * (2 * n))()
    total, wsb = C.c_int64(0), C.c_size_t(0)
    _check(lib.vqa_qwen_preprocess_plan(H, W, n, patch, merge, min_pixels, max_pixels, grid, C.byref(total), C.byref(wsb)), None,
           "vqa_qwen_preprocess_plan")
    return [(1, int(grid[2 * i]), int(grid[2 * i + 1])) for i in range(n)], int(total.value), int(wsb.value)


def qwen_preprocess_u8(images: Sequence[torch.Tensor], device, patch: int = 14, temporal_patch: int = 2, merge: int = 2,
                       min_pixels: int = 56 * 56, max_pixels: int = 14 * 14 * 4 * 1280, mean=CLIP_MEAN, std=CLIP_STD,
                       out_dtype: torch.dtype = torch.float32):
    """Decoded still images (uint8 HWC RGB, host or device) -> (pixel_patches [sum gh*gw, 3*temporal*patch^2] on the device,
    [(1, gh, gw), ...]) by ONE kernel launch: smart_resize + PIL-exact bicubic + /255 + normalise + frame duplication + merge-order
    patch rows -- bit-identical to models/vqascore_models/qwen_utils.qwen_image_to_patches (the CPU path)."""
    lib = _lib.load()
    dev = torch.device(device)
    n = len(images)
    assert n > 0
    hs, ws, offs, total = [], [], [], 0
    for im in images:
        assert im.dtype == torch.uint8 and im.dim() == 3 and im.shape[2] == 3, "images must be uint8 [h, w, 3]"
        hs.append(int(im.shape[0])); ws.append(int(im.shape[1])); offs.append(total)
        total += int(im.numel())
    grids, rows, need = qwen_preprocess_plan(list(zip(hs, ws)), patch, merge, min_pixels, max_pixels)
    if isinstance(images, torch.Tensor):
        src = images.contiguous().view(-1)
        src = src if src.is_cuda else src.to(dev, non_blocking=True)
    elif all(im.is_cuda for im in images):
        src = images[0].contiguous().view(-1) if n == 1 else torch.cat([im.contiguous().view(-1) for im in images])
    else:
        stage = torch.empty(total, dtype=torch.uint8, pin_memory=True)
        for im, o in zip(images, offs):
            stage[o:o + im.numel()] = im.contiguous().view(-1)
        src = stage.to(dev, non_blocking=True)
    out = torch.empty(rows, 3 * temporal_patch * patch * patch, dtype=out_dtype, device=dev)
    wsb = torch.empty(max(need, 16), dtype=torch.uint8, device=dev)
    ring = _staging(dev)
    stage_buf = ring.acquire(wsb.numel())
    with torch.cuda.device(dev):
        rc = lib.vqa_qwen_preprocess(_ptr(src), (C.c_int64 * n)(*offs), (C.c_int32 * n)(*hs), (C.c_int32 * n)(*ws), n, patch, temporal_patch,
                                     merge, min_pixels, max_pixels, (C.c_float * 3)(*mean), (C.c_float * 3)(*std), _ptr(out),
                                     _lib.VQA_DTYPE_F32 if out_dtype == torch.float32 else _lib.VQA_DTYPE_BF16, _ptr(wsb), wsb.numel(),
                                     stage_buf.data_ptr(), _stream_ptr(dev))
    ring.release(dev)
    _check(rc, None, "vqa_qwen_preprocess")
    return out, grids


def _video_arrays(videos, policies, min_pixels, max_pixels):
    n = len(videos)
    assert n > 0 and len(policies) == n and len(min_pixels) == n and len(max_pixels) == n
    fs, hs, ws, offs, total = [], [], [], [], 0
    for v in videos:
        assert v.dtype == torch.uint8 and v.dim() == 4 and v.shape[3] == 3, "videos must be uint8 [frames, h, w, 3]"
        fs.append(int(v.shape[0])); hs.append(int(v.shape[1])); ws.append(int(v.shape[2])); offs.append(total)
        total += int(v.numel())
    i32 = lambda xs: (C.c_int32 * n)(*[int(x) for x in xs])
    i64 = lambda xs: (C.c_int64 * n)(*[int(x) for x in xs])
    return dict(F=i32(fs), H=i32(hs), W=i32(ws), P=i32(policies), MN=i64(min_pixels), MX=i64(max_pixels), O=i64(offs), total=total)


def qwen_video_preprocess_plan(sizes_fhw: Sequence[Sequence[int]], policies: Sequence[int], min_pixels: Sequence[int],
                               max_pixels: Sequence[int], patch: int = 14, temporal_patch: int = 2, merge: int = 2):
    """Host-only geometry of the Qwen video pre-processing: (frames, h, w) per video -> ([(t, gh, gw), ...], total patch rows,
    workspace bytes)."""
    lib = _lib.load()
    n = len(sizes_fhw)
    a = _video_arrays([torch.empty(int(f), int(h), int(w), 3, dtype=torch.uint8, device="meta") for f, h, w in sizes_fhw], policies,
                      min_pixels, max_pixels)
    grid = (C.c_int32 * (3 * n))()
    total, wsb = C.c_int64(0), C.c_size_t(0)
    _check(lib.vqa_qwen_video_preprocess_plan(a["H"], a["W"], a["F"], a["P"], n, patch, temporal_patch, merge, a["MN"], a["MX"], grid,
                                              C.byref(total), C.byref(wsb)), None, "vqa_qwen_video_preprocess_plan")
    return [tuple(int(grid[3 * i + k]) for k in range(3)) for i in range(n)], int(total.value), int(wsb.value)


def qwen_video_preprocess_u8(videos: Sequence[torch.Tensor], policies: Sequence[int], device, min_pixels: Sequence[int],
                             max_pixels: Sequence[int], patch: int = 14, temporal_patch: int = 2, merge: int = 2, mean=CLIP_MEAN,
                             std=CLIP_STD, out_dtype: torch.dtype = torch.float32):
    """Sampled video frames (uint8 [frames, h, w, 3] RGB per video, host or device) -> (pixel_patches [sum t*gh*gw, 3*tp*patch^2] on
    the device, [(t, gh, gw), ...]) by ONE kernel launch over every frame of every video: per-video smart_resize with its own pixel
    bounds, the resample of `policies[v]` (_lib.VQA_RESAMPLE_PIL for frame stacks, _lib.VQA_RESAMPLE_TORCHVISION for decoded files),
    /255, normalise, temporal pairing (an odd last frame fills both slots of its pair) and merge-order rows. Bit-identical to
    qwen_utils.qwen_video_to_patches of pil_resize_frames / torchvision_resize_u8 (the latter up to fp32 ties, see
    vqa_resample_table_tv)."""
    lib = _lib.load()
    dev = torch.device(device)
    n = len(videos)
    a = _video_arrays(videos, policies, min_pixels, max_pixels)
    grid = (C.c_int32 * (3 * n))()
    rows, need = C.c_int64(0), C.c_size_t(0)
    _check(lib.vqa_qwen_video_preprocess_plan(a["H"], a["W"], a["F"], a["P"], n, patch, temporal_patch, merge, a["MN"], a["MX"], grid,
                                              C.byref(rows), C.byref(need)), None, "vqa_qwen_video_preprocess_plan")
    grids = [tuple(int(grid[3 * i + k]) for k in range(3)) for i in range(n)]
    if all(v.is_cuda for v in videos):
        src = videos[0].contiguous().view(-1) if n == 1 else torch.cat([v.contiguous().view(-1) for v in videos])
    else:
        stage = torch.empty(a["total"], dtype=torch.uint8, pin_memory=True)
        o = 0
        for v in videos:
            stage[o:o + v.numel()] = v.contiguous().view(-1).cpu()
            o += v.numel()
        src = stage.to(dev, non_blocking=True)
    out = torch.empty(int(rows.value), 3 * temporal_patch * patch * patch, dtype=out_dtype, device=dev)
    wsb = torch.empty(max(int(need.value), 16), dtype=torch.uint8, device=dev)
    ring = _staging(dev)
    stage_buf = ring.acquire(wsb.numel())
    with torch.cuda.device(dev):
        rc = lib.vqa_qwen_video_preprocess(_ptr(src), a["O"], a["H"], a["W"], a["F"], a["P"], n, patch, temporal_patch, merge, a["MN"],
                                           a["MX"], (C.c_float * 3)(*mean), (C.c_float * 3)(*std), _ptr(out),
                                           _lib.VQA_DTYPE_F32 if out_dtype == torch.float32 else _lib.VQA_DTYPE_BF16, _ptr(wsb),
                                           wsb.numel(), stage_buf.data_ptr(), _stream_ptr(dev))
    ring.release(dev)
    _check(rc, None, "vqa_qwen_video_preprocess")
    return out, grids


def resample_table_tv(in_size: int, out_size: int):
    """Host-only: (bounds int32 [out, 2], taps fp32 [out, ksize], fma) of one axis of the torchvision-policy resize, as the kernel uses
    them (vqa_resample_table_tv)."""
    lib = _lib.load()
    fma = C.c_int32(0)
    ks = int(lib.vqa_resample_table_tv(in_size, out_size, 0, out_size, None, None, C.byref(fma)))
    if ks == 0:
        raise ValueError(_lib.last_error(None))
    bounds = torch.zeros(out_size, 2, dtype=torch.int32)
    taps = torch.zeros(out_size, ks, dtype=torch.float32)
    lib.vqa_resample_table_tv(in_size, out_size, 0, out_size, C.cast(bounds.data_ptr(), C.POINTER(C.c_int32)),
                              C.cast(taps.data_ptr(), C.POINTER(C.c_float)), C.byref(fma))
    return bounds, taps, bool(fma.value)


# ================================================================================================ Qwen2.5-VL
def convert_qwen_state_dict(sd: Dict[str, torch.Tensor], cfg, device) -> Dict[str, torch.Tensor]:
    """HF `Qwen2_5_VLForConditionalGeneration` names -> the engine's fused bf16 layout:
      * vision qkv / proj: the HF tensors as they are ([3*H*hd, Dv] rows ordered (q|k|v, head, dim); [Dv, H*hd]). The qkv GEMM's epilogue
        scatters each 80-wide head into the 128-wide slots of the packed activation [L, 3*H*128] the attention kernel reads (pad columns
        zeroed once per forward), the attention kernel writes compact heads [L, H*hd];
      * vision gate|up rows concatenated with the MLP width zero-padded to a multiple of 128; down-projection columns padded;
      * language-model q|k|v rows concatenated (+ biases), gate|up rows concatenated."""
    out: Dict[str, torch.Tensor] = {}

    def put(name, t):
        out[name] = t.detach().to(device=device, dtype=torch.bfloat16).contiguous()

    v = "model.visual."
    Dv, H, hd = cfg.vit_hidden, cfg.vit_heads, cfg.vit_head_dim
    mp = cfg.vit_mlp_padded
    put("vis.patch_embed", sd[v + "patch_embed.proj.weight"].reshape(Dv, -1))
    for l in range(cfg.vit_depth):
        p, q = v + f"blocks.{l}.", f"vis.{l}."
        put(q + "norm1", sd[p + "norm1.weight"]); put(q + "norm2", sd[p + "norm2.weight"])
        # HF's fused qkv rows are already ordered (q|k|v, head, dim) and proj's columns (head, dim): bound as they are, at the native head width
        put(q + "qkv.weight", sd[p + "attn.qkv.weight"]); put(q + "qkv.bias", sd[p + "attn.qkv.bias"])
        put(q + "proj.weight", sd[p + "attn.proj.weight"]); put(q + "proj.bias", sd[p + "attn.proj.bias"])
        gu = torch.zeros(2 * mp, Dv); gb = torch.zeros(2 * mp)
        gu[: cfg.vit_mlp] = sd[p + "mlp.gate_proj.weight"].float(); gu[mp: mp + cfg.vit_mlp] = sd[p + "mlp.up_proj.weight"].float()
        gb[: cfg.vit_mlp] = sd[p + "mlp.gate_proj.bias"].float(); gb[mp: mp + cfg.vit_mlp] = sd[p + "mlp.up_proj.bias"].float()
        put(q + "gate_up.weight", gu); put(q + "gate_up.bias", gb)
        dw = torch.zeros(Dv, mp); dw[:, : cfg.vit_mlp] = sd[p + "mlp.down_proj.weight"].float()
        put(q + "down.weight", dw); put(q + "down.bias", sd[p + "mlp.down_proj.bias"])
    put("vis.merger.ln_q", sd[v + "merger.ln_q.weight"])
    put("vis.merger.fc1.weight", sd[v + "merger.mlp.0.weight"]); put("vis.merger.fc1.bias", sd[v + "merger.mlp.0.bias"])
    put("vis.merger.fc2.weight", sd[v + "merger.mlp.2.weight"]); put("vis.merger.fc2.bias", sd[v + "merger.mlp.2.bias"])
    t = "model.language_model."
    put("llm.embed", sd[t + "embed_tokens.weight"])
    put("llm.norm", sd[t + "norm.weight"])
    put("llm.lm_head", sd["lm_head.weight"])
    for l in range(cfg.layers):
        p, q = t + f"layers.{l}.", f"llm.{l}."
        put(q + "ln1", sd[p + "input_layernorm.weight"]); put(q + "ln2", sd[p + "post_attention_layernorm.weight"])
        put(q + "qkv.weight", torch.cat([sd[p + f"self_attn.{n}_proj.weight"] for n in "qkv"], dim=0))
        put(q + "qkv.bias", torch.cat([sd[p + f"self_attn.{n}_proj.bias"] for n in "qkv"], dim=0))
        put(q + "o.weight", sd[p + "self_attn.o_proj.weight"])
        put(q + "gate_up.weight", torch.cat([sd[p + "mlp.gate_proj.weight"], sd[p + "mlp.up_proj.weight"]], dim=0))
        put(q + "down.weight", sd[p + "mlp.down_proj.weight"])
    return out


class QwenVLEngine:
    """Qwen2.5-VL VQAScore engine: P(answer token | image, prompt) for a whole batch of prompts in one prefill."""

    def __init__(self, cfg, device="cuda:0", emulate_bf16_rounding: bool = True):
        from . import qwen_host
        if not torch.cuda.is_available():
            raise RuntimeError("QwenVLEngine needs a CUDA device (sm_100a); there is no CPU path")
        if cfg.head_dim != 128:
            raise ValueError("the language-model attention kernel is specialised for head_dim == 128")
        self.lib = _lib.load()
        self.cfg = cfg
        self.device = torch.device(device)
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        mask = 0
        for l in cfg.fullatt_block_indexes:
            mask |= 1 << l
        c = _lib.VqaQwen25VLConfig(vit_depth=cfg.vit_depth, vit_hidden=cfg.vit_hidden, vit_heads=cfg.vit_heads,
                                   vit_head_dim=cfg.vit_head_dim, vit_mlp=cfg.vit_mlp, patch_dim=cfg.patch_dim,
                                   spatial_merge=cfg.spatial_merge_size, out_hidden=cfg.out_hidden, fullatt_mask=mask,
                                   hidden=cfg.hidden, layers=cfg.layers, heads=cfg.heads, kv_heads=cfg.kv_heads, mlp=cfg.mlp,
                                   vocab=cfg.vocab, rms_eps=cfg.rms_eps, emulate_bf16_rounding=1 if emulate_bf16_rounding else 0)
        self._h = C.c_void_p()
        with torch.cuda.device(idx):
            _check(self.lib.vqa_create_qwen25vl(C.byref(c), idx, C.byref(self._h)), None, "vqa_create_qwen25vl")
        t_inv, t_axis, v_inv, v_axis = qwen_host.rope_tables(cfg.head_dim, cfg.rope_theta, cfg.mrope_section, cfg.vit_head_dim)
        fp = lambda t: t.numpy().ctypes.data_as(C.POINTER(C.c_float))
        ip = lambda t: t.numpy().ctypes.data_as(C.POINTER(C.c_int32))
        _check(self.lib.vqa_qwen25vl_set_rope(self._h, fp(t_inv), ip(t_axis), t_inv.numel(), fp(v_inv), ip(v_axis), v_inv.numel()),
               self._h, "vqa_qwen25vl_set_rope")
        self._weights: Dict[str, torch.Tensor] = {}
        self._workspace: Optional[torch.Tensor] = None
        self._vision_cache: "collections.OrderedDict[tuple, dict]" = collections.OrderedDict()   # per-batch index sets, LRU-bounded

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            self.lib.vqa_destroy(h)
            self._h = C.c_void_p()

    bind_engine_tensors = ClipT5Engine.bind_engine_tensors
    last_launch_count = ClipT5Engine.last_launch_count
    set_profile = ClipT5Engine.set_profile
    read_profile = ClipT5Engine.read_profile

    def load_state_dict(self, sd: Dict[str, torch.Tensor]):
        self.bind_engine_tensors(convert_qwen_state_dict(sd, self.cfg, self.device))

    def vision_indices(self, grid_thw):
        """Window order, rotary positions and cumulative lengths for a list of (t, h, w) grids; cached per grid tuple."""
        from . import qwen_host
        key = tuple(tuple(int(x) for x in g) for g in grid_thw)
        hit = self._vision_cache.get(key)
        if hit is not None:
            self._vision_cache.move_to_end(key)
            return hit
        cfg, dev = self.cfg, self.device
        merge, unit = cfg.spatial_merge_size, cfg.spatial_merge_size ** 2
        widx, cu_win, cu_frames = qwen_host.vision_window_index(key, merge, cfg.window_size, cfg.patch_size)
        pos = qwen_host.vision_rot_pos_ids(key, merge)                                   # [L, 2] processor order
        L = pos.shape[0]
        pos_win = pos.reshape(L // unit, unit, 2)[widx].reshape(L, 2)                    # window order (:478-484)
        i32 = lambda t: t.to(torch.int32).contiguous().to(dev)
        out = dict(window_index=i32(widx), reverse_index=i32(torch.argsort(widx)), vis_pos_hw=i32(pos_win.t()),
                   cu_window=i32(cu_win), cu_frames=i32(cu_frames), n_windows=cu_win.numel() - 1, n_frames=cu_frames.numel() - 1,
                   max_window=int((cu_win[1:] - cu_win[:-1]).max()), max_frame=int((cu_frames[1:] - cu_frames[:-1]).max()),
                   n_patches=L)
        self._vision_cache[key] = out
        while len(self._vision_cache) > 64:          # a dataset with varied image sizes makes a new key per batch: keep the device memory bounded
            self._vision_cache.popitem(last=False)
        return out

    def score_tensors(self, pixel_patches: torch.Tensor, grid_thw, input_ids: torch.Tensor, seq_lens: torch.Tensor,
                      feat_index: torch.Tensor, position_ids: torch.Tensor, answer_ids: torch.Tensor, temperature: float = 1.0,
                      out: Optional[torch.Tensor] = None, return_logprobs: bool = False, repetition_penalty: float = 1.0):
        """pixel_patches [sum P, patch_dim] fp32/bf16 cuda; grid_thw list of (t,h,w); the int32 cuda tensors come from
        qwen_host.build_batch_indices. repetition_penalty != 1 applies HF's RepetitionPenaltyLogitsProcessor over each sample's
        prompt ids before the softmax (what `generate(..., output_scores=True)` returns when the checkpoint's
        generation_config.json carries one, SURVEY F8). Returns probabilities [B] fp32 on the device."""
        dev = self.device
        vi = self.vision_indices(grid_thw)
        assert pixel_patches.is_cuda and pixel_patches.is_contiguous() and pixel_patches.shape == (vi["n_patches"], self.cfg.patch_dim)
        assert pixel_patches.dtype in (torch.float32, torch.bfloat16)
        for t in (input_ids, seq_lens, feat_index, position_ids, answer_ids):
            assert t.is_cuda and t.dtype == torch.int32 and t.is_contiguous()
        B, S = input_ids.shape
        need = int(self.lib.vqa_qwen25vl_workspace_bytes(self._h, B, S, vi["n_patches"]))
        if self._workspace is None or self._workspace.numel() < need:
            self._workspace = None
            self._workspace = torch.empty(need, dtype=torch.uint8, device=dev)
        if out is None:
            out = torch.empty(B, dtype=torch.float32, device=dev)
        logp = torch.empty(B, dtype=torch.float32, device=dev) if return_logprobs else None
        pdt = _lib.VQA_DTYPE_F32 if pixel_patches.dtype == torch.float32 else _lib.VQA_DTYPE_BF16
        with torch.cuda.device(dev):
            rc = self.lib.vqa_qwen25vl_score(self._h, _ptr(pixel_patches), pdt, vi["n_patches"], _ptr(vi["vis_pos_hw"]),
                                             _ptr(vi["window_index"]), _ptr(vi["reverse_index"]), _ptr(vi["cu_window"]), vi["n_windows"],
                                             vi["max_window"], _ptr(vi["cu_frames"]), vi["n_frames"], vi["max_frame"], _ptr(input_ids),
                                             _ptr(seq_lens), _ptr(feat_index), _ptr(position_ids), _ptr(answer_ids), B, S,
                                             float(temperature), float(repetition_penalty), _ptr(out), _ptr(logp), _ptr(self._workspace),
                                             self._workspace.numel(), _stream_ptr(dev))
        _check(rc, self._h, "vqa_qwen25vl_score")
        self._last_call = (B, B * S, vi["n_patches"])       # what topk_last() needs to find the final hidden states again
        return (out, logp) if return_logprobs else out

    def topk_last(self, k: int = 5, temperature: float = 1.0, repetition_penalty: float = 1.0):
        """Top-k next tokens (ids [B, k] int32, probabilities [B, k] fp32, most probable first) of the prompts of the LAST score_tensors /
        score_prompts call, under the same logit processing as the scores -- the reference's forward_with_trace output
        (qwen2vl_model.py:439-447). Trace mode only: materialises the last position's [B, vocab] logits in the workspace."""
        if getattr(self, "_last_call", None) is None:
            raise RuntimeError("topk_last() follows a scoring call")
        B, rows, n_patches = self._last_call
        dev = self.device
        ids = torch.empty(B, k, dtype=torch.int32, device=dev)
        probs = torch.empty(B, k, dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            rc = self.lib.vqa_qwen25vl_topk(self._h, B, rows, n_patches, k, float(temperature), float(repetition_penalty), _ptr(ids), _ptr(probs),
                                            _ptr(self._workspace), self._workspace.numel(), _stream_ptr(dev))
        _check(rc, self._h, "vqa_qwen25vl_topk")
        return ids, probs

    def debug_tensors(self, batch: int, seq_len: int, n_patches: int) -> Dict[str, torch.Tensor]:
        """Views into the workspace of the LAST call with these sizes (synchronise first). Parity investigations only."""
        off = (C.c_size_t * 4)()
        _check(self.lib.vqa_qwen25vl_debug_layout(self._h, batch, seq_len, n_patches, off, 4), self._h, "vqa_qwen25vl_debug_layout")
        cfg, ws = self.cfg, self._workspace
        unit = cfg.spatial_merge_size ** 2

        def view(o, rows, cols):
            return ws[o:o + rows * cols * 2].view(torch.bfloat16).view(rows, cols)
        return dict(last_hidden=view(off[0], batch, cfg.hidden), vision_feats=view(off[1], n_patches // unit, cfg.out_hidden))

    def score_packed(self, pixel_patches: torch.Tensor, grid_thw, packed: Dict[str, torch.Tensor], answer_ids: torch.Tensor,
                     temperature: float = 1.0, repetition_penalty: float = 1.0, out: Optional[torch.Tensor] = None):
        """One prefill over PACKED rows (qwen_host.build_packed_indices, tensors already on the device): prompts over the same image share
        the K/V of their [chat prefix + vision tokens]."""
        dev = self.device
        vi = self.vision_indices(grid_thw)
        assert pixel_patches.is_cuda and pixel_patches.is_contiguous() and pixel_patches.shape == (vi["n_patches"], self.cfg.patch_dim)
        B, R = int(answer_ids.numel()), int(packed["total_rows"])
        need = int(self.lib.vqa_qwen25vl_packed_workspace_bytes(self._h, B, R, vi["n_patches"]))
        if self._workspace is None or self._workspace.numel() < need:
            self._workspace = None
            self._workspace = torch.empty(need, dtype=torch.uint8, device=dev)
        if out is None:
            out = torch.empty(B, dtype=torch.float32, device=dev)
        pdt = _lib.VQA_DTYPE_F32 if pixel_patches.dtype == torch.float32 else _lib.VQA_DTYPE_BF16
        with torch.cuda.device(dev):
            rc = self.lib.vqa_qwen25vl_score_packed(
                self._h, _ptr(pixel_patches), pdt, vi["n_patches"], _ptr(vi["vis_pos_hw"]), _ptr(vi["window_index"]), _ptr(vi["reverse_index"]),
                _ptr(vi["cu_window"]), vi["n_windows"], vi["max_window"], _ptr(vi["cu_frames"]), vi["n_frames"], vi["max_frame"],
                _ptr(packed["input_ids"]), _ptr(packed["feat_index"]), _ptr(packed["position_ids"]), R, _ptr(packed["cu_seqlens"]),
                _ptr(packed["kv_prefix"]), int(packed["n_seq"]), int(packed["max_seq_len"]), _ptr(packed["pair_row"]), _ptr(packed["pair_seq"]),
                _ptr(answer_ids), B, int(packed["max_prompt_len"]), float(temperature), float(repetition_penalty), _ptr(out), None,
                _ptr(self._workspace), self._workspace.numel(), _stream_ptr(dev))
        _check(rc, self._h, "vqa_qwen25vl_score_packed")
        self._last_call = (B, R, vi["n_patches"])
        return out

    def score_prompts(self, pixel_patches, grid_thw, prompts, answer_ids, image_of_sample=None, temperature: float = 1.0,
                      repetition_penalty: float = 1.0, second_per_grid_ts=None, share_prefix: Optional[bool] = None):
        """Convenience: prompts = list of 1-D id lists (each with one image- or video-token run). Host index logic + one engine
        call. Videos are grids with t > 1 whose prompt run uses cfg.video_token_id (second_per_grid_ts = temporal_patch / fps).
        share_prefix: None = automatically when at least two prompts start with the same [chat prefix + vision run] over the same image
        (the M x N scoring API repeats every image N times, reference score.py:104-106); their prefix then runs through the language
        model once (KV-prefix sharing, exact under causal attention)."""
        from . import qwen_host
        cfg, dev = self.cfg, self.device
        B = len(prompts)
        img = list(image_of_sample) if image_of_sample is not None else list(range(B))
        if share_prefix is None or share_prefix:
            pk = qwen_host.build_packed_indices([list(map(int, p)) for p in prompts], [tuple(map(int, g)) for g in grid_thw], img,
                                                cfg.image_token_id, cfg.spatial_merge_size, cfg.tokens_per_second,
                                                video_token_id=cfg.video_token_id, second_per_grid_ts=second_per_grid_ts)
            if pk["n_shared"] > 0 or share_prefix:
                d = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in pk.items()}
                ans = torch.as_tensor(list(map(int, answer_ids)), dtype=torch.int32).to(dev)
                return self.score_packed(pixel_patches.to(dev), grid_thw, d, ans, temperature, repetition_penalty)
        idx = qwen_host.build_batch_indices([list(map(int, p)) for p in prompts], [tuple(map(int, g)) for g in grid_thw], img,
                                            cfg.image_token_id, cfg.spatial_merge_size, cfg.tokens_per_second,
                                            video_token_id=cfg.video_token_id, second_per_grid_ts=second_per_grid_ts)
        d = {k: v.to(dev) for k, v in idx.items()}
        ans = torch.as_tensor(list(map(int, answer_ids)), dtype=torch.int32).to(dev)
        return self.score_tensors(pixel_patches.to(dev), grid_thw, d["input_ids"], d["seq_lens"], d["feat_index"], d["position_ids"],
                                  ans, temperature, repetition_penalty=repetition_penalty)
