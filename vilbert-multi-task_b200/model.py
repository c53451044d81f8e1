"""VILBertForVLTasks: the object protocol of the reference worker on top of the C ABI.

    config = BertConfig.from_json_file(path)                                   worker.py:495, 506
    model  = VILBertForVLTasks.from_pretrained(ckpt, config=config,
                                               num_labels=3129, default_gpu=True)   worker.py:530-532
    model.eval(); model.cuda(0)                                                worker.py:534-536
    out10  = model(question, features, spatials, segment_ids, input_mask, image_mask,
                   co_attention_mask, task_tokens, output_all_attention_masks=True)  worker.py:286-289

Everything between the input tensors and the ten outputs runs in libvilbert_b200.so (hand-written sm_100a
kernels).  torch is used only as the tensor container and for the CUDA stream.  No CPU path exists: calling
the model without a B200 raises.
"""
from __future__ import annotations

import ctypes as C
import json
from typing import Dict, Optional

import torch

from . import _lib as L
from .config import BertConfig

_DTYPES = {torch.float32: L.F32, torch.float16: L.F16, torch.bfloat16: L.BF16}


def _normalise_state_dict(sd) -> Dict[str, torch.Tensor]:
    if isinstance(sd, dict) and "state_dict" in sd and isinstance(sd["state_dict"], dict):
        sd = sd["state_dict"]
    if isinstance(sd, dict) and "model_state_dict" in sd and isinstance(sd["model_state_dict"], dict):
        sd = sd["model_state_dict"]
    out = {}
    for k, v in sd.items():
        if not torch.is_tensor(v):
            continue
        if v.dtype in (torch.int64, torch.int32, torch.bool) or v.dim() == 0 or v.dim() > 2:
            continue                      # e.g. position_ids buffers, num_batches_tracked
        if v.dtype not in _DTYPES:
            v = v.float()
        out[k] = v.detach().cpu().contiguous()
    return out


class VILBertForVLTasks(object):
    """Drop-in for ``vilbert.vilbert.VILBertForVLTasks`` on the inference path the worker uses."""

    def __init__(self, config: BertConfig, num_labels: int = 3129, state_dict=None, default_gpu: bool = True,
                 use_cuda_graph: bool = True, use_pdl: Optional[bool] = None, strict: bool = True, compute_dtype: str = "fp16",
                 fused_layernorm: bool = False, return_attention: bool = False, max_plans: int = 0, ln_fold: bool = False):
        self.config = config
        self.num_labels = num_labels
        self._sd = _normalise_state_dict(state_dict) if state_dict is not None else None
        self._handle = None
        self._device = None
        if compute_dtype not in ("fp16", "bf16", "fp32x"):
            raise ValueError("compute_dtype must be 'fp16', 'bf16' or 'fp32x'")
        # Format of the tensor-core operands (weights and activations): fp16 (default), bf16, or "fp32x" -- the fp32-parity mode:
        # every operand as an fp16 hi/lo pair, three tensor-core products per k-step, fp32 attention (<= 1e-3 per logit against
        # the reference's fp32 forward, 3x the tensor work).  Accumulation, residual stream, LayerNorm, softmax and logits are
        # fp32 in every mode.
        self._opts = dict(use_cuda_graph=use_cuda_graph, use_pdl=use_pdl, strict=strict, compute_dtype=compute_dtype,
                          fused_layernorm=fused_layernorm, max_plans=int(max_plans), ln_fold=bool(ln_fold))
        # attn_data_list (element 9 of the tuple): the reference returns the 24 layers' attention probabilities when called with
        # output_all_attention_masks=True (worker.py:287-288) and never reads them; here they are computed only when this flag
        # is set as well (model.return_attention = True), otherwise element 9 is [].
        self.return_attention = bool(return_attention)
        self.training = False
        self._dims = {}

    # ------------------------------------------------------------------ reference construction protocol
    @classmethod
    def from_pretrained(cls, pretrained_model_name_or_path, config=None, num_labels=3129, default_gpu=True,
                        state_dict=None, **kwargs):
        if config is None:
            raise ValueError("config is required (worker.py:530-532 always passes it)")
        if state_dict is None:
            if isinstance(pretrained_model_name_or_path, dict):
                state_dict = pretrained_model_name_or_path
            else:
                state_dict = torch.load(pretrained_model_name_or_path, map_location="cpu")
        return cls(config, num_labels=num_labels, state_dict=state_dict, default_gpu=default_gpu, **kwargs)

    def eval(self):
        self.training = False
        return self

    def train(self, mode: bool = True):
        if mode:
            raise L.VilbertB200Error("vilbert_b200 is an inference engine; train() is not supported")
        return self

    def cuda(self, device=0):
        if isinstance(device, torch.device):
            device = device.index or 0
        device = 0 if device is None else int(device)
        if self._handle is not None and self._device == device:
            return self
        self._create(device)
        return self

    def to(self, device):
        device = torch.device(device)
        if device.type != "cuda":
            raise L.VilbertB200Error("vilbert_b200 runs on sm_100 GPUs only; there is no CPU path")
        return self.cuda(device.index or 0)

    def half(self):            # tensor-core operands are 16-bit already (compute_dtype); accepted for call-site compatibility
        return self

    def parameters(self):
        return iter(())

    def state_dict(self):
        return dict(self._sd) if self._sd is not None else {}

    # ------------------------------------------------------------------ engine lifetime
    def _config_json(self) -> bytes:
        d = {k: v for k, v in self.config.to_dict().items()
             if isinstance(v, (int, float, str, bool, list)) or v is None}
        return json.dumps(d).encode()

    def _create(self, device: int):
        lib = L.load()
        if self._sd is None:
            raise L.VilbertB200Error("no state_dict: build the model with from_pretrained(...)")
        if not torch.cuda.is_available():
            raise L.VilbertB200Error("no CUDA device visible; vilbert_b200 has no CPU fallback")
        self.close()
        names = [k.encode() for k in self._sd]
        arr = (L.Tensor * len(self._sd))()
        keep = []
        for i, (k, v) in enumerate(self._sd.items()):
            t = arr[i]
            t.name = names[i]
            t.dtype = _DTYPES[v.dtype]
            t.ndim = v.dim()
            t.shape[0] = v.shape[0]
            t.shape[1] = v.shape[1] if v.dim() == 2 else 0
            t.data = v.data_ptr()
            keep.append(v)
        opt = L.Options()
        opt.device = device
        opt.num_labels = int(self.num_labels or 0)
        opt.use_cuda_graph = 1 if self._opts["use_cuda_graph"] else -1
        # None: engine default (programmatic dependent launch on every kernel); True: the same, forced; False: none
        opt.use_pdl = 0 if self._opts["use_pdl"] is None else (1 if self._opts["use_pdl"] else -1)
        opt.strict = 1 if self._opts["strict"] else -1
        opt.act_fp16 = -1 if self._opts["compute_dtype"] == "bf16" else 1
        opt.fused_layernorm = 1 if self._opts["fused_layernorm"] else 0
        opt.split_fp32 = 1 if self._opts["compute_dtype"] == "fp32x" else 0
        opt.max_plans = self._opts["max_plans"]
        opt.ln_fold = 1 if self._opts["ln_fold"] else 0
        h = C.c_void_p()
        with torch.cuda.device(device):
            rc = lib.vb200_create(self._config_json(), len(self._sd), arr, C.byref(opt), C.byref(h))
        L.check(rc, None)
        self._handle, self._device = h, device
        for key in ("hidden_size", "v_hidden_size", "bi_hidden_size", "vocab_size", "v_target_size",
                    "v_feature_size", "num_labels", "gqa_labels", "task_specific_tokens", "weight_bytes",
                    "operand_width_factor"):
            v = C.c_int64()
            L.check(lib.vb200_model_dim(h, key.encode(), C.byref(v)), h)
            self._dims[key] = v.value

    def close(self):
        if self._handle is not None:
            L.load().vb200_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ forward
    def _out_shapes(self, B, T, V, select):
        d = self._dims
        shapes = {
            "vil_prediction": (L.OUT_VIL_PREDICTION, (B, d["num_labels"])),
            "vil_prediction_gqa": (L.OUT_VIL_PREDICTION_GQA, (B, d["gqa_labels"])),
            "vil_logit": (L.OUT_VIL_LOGIT, (B, 1)),
            "vil_binary_prediction": (L.OUT_VIL_BINARY_PREDICTION, (B // 2, 2) if B % 2 == 0 else (B, 2)),
            "vil_tri_prediction": (L.OUT_VIL_TRI_PREDICTION, (B, 3)),
            "vision_prediction": (L.OUT_VISION_PREDICTION, (B, V, d["v_target_size"])),
            "vision_logit": (L.OUT_VISION_LOGIT, (B, V, 1)),
            "linguisic_prediction": (L.OUT_LINGUISIC_PREDICTION, (B, T, d["vocab_size"])),
            "linguisic_logit": (L.OUT_LINGUISIC_LOGIT, (B, T, 1)),
        }
        return {k: s for k, (bit, s) in shapes.items() if select & bit}

    def plan_info(self, batch, n_tokens, n_regions, select=L.OUT_TASK_HEADS):
        n, f = C.c_int64(), C.c_double()
        L.check(L.load().vb200_plan_info(self._handle, batch, n_tokens, n_regions, select, C.byref(n), C.byref(f)),
                self._handle)
        return n.value, f.value

    def set_option(self, key, value):
        """Run-time knobs of the engine (include/vilbert_b200.h, vb200_set_option): "max_plans", "chain_ffn", "prune_tail",
        "profile_grid_pct"."""
        L.check(L.load().vb200_set_option(self._handle, key.encode(), int(value)), self._handle)

    def profile_ops(self, batch, n_tokens, n_regions, select=L.OUT_TASK_HEADS, iters=5, grid_pct=0):
        """Per-launch device times (ms) of one forward: every kernel replayed alone from its own CUDA graph between two events.
        grid_pct (10..100): persistent-grid size of the GEMMs for THIS measurement only (production: 2/3 of the CTA slots)."""
        if grid_pct:
            L.check(L.load().vb200_set_option(self._handle, b"profile_grid_pct", int(grid_pct)), self._handle)
        cap = 2048
        n = C.c_int32()
        kinds = (C.c_int32 * cap)()
        ms = (C.c_double * cap)()
        fl = (C.c_double * cap)()
        dims = (C.c_int32 * (4 * cap))()
        L.check(L.load().vb200_profile_ops(self._handle, batch, n_tokens, n_regions, select, iters, cap, C.byref(n), kinds, ms,
                                           fl, dims), self._handle)
        names = {0: "gemm", 1: "self_attention", 2: "co_attention", 3: "rowdot", 4: "layernorm", 5: "attention_f32"}
        return [dict(kind=names.get(kinds[i], "?"), ms=ms[i], flops=fl[i], dims=list(dims[4 * i:4 * i + 4]))
                for i in range(min(n.value, cap))]

    def _prep(self, question, features, spatials, segment_ids, input_mask, image_mask, task_tokens, device):
        def dev(t, dtype):
            if not torch.is_tensor(t):
                t = torch.as_tensor(t)
            if t.dtype != dtype:
                t = t.to(dtype)
            if t.device != device:
                t = t.to(device, non_blocking=True)
            return t.contiguous()
        B, Tin = question.shape
        V = features.shape[1]
        q = dev(question, torch.int64)
        f = dev(features, torch.float32)
        s = dev(spatials, torch.float32)
        seg = dev(segment_ids if segment_ids is not None else torch.zeros_like(question), torch.int64)
        im = dev(input_mask if input_mask is not None else torch.ones_like(question), torch.int64)
        vm = dev(image_mask if image_mask is not None else torch.ones(B, V, dtype=torch.uint8), torch.uint8)
        if task_tokens is None:
            task_tokens = torch.zeros(B, 1, dtype=torch.int64)
        tk = dev(task_tokens, torch.int64).reshape(B, -1)[:, :1].contiguous()
        if tuple(f.shape) != (B, V, self._dims["v_feature_size"]) or tuple(s.shape) != (B, V, 5) \
                or tuple(seg.shape) != (B, Tin) or tuple(im.shape) != (B, Tin) or tuple(vm.shape) != (B, V):
            raise ValueError("input shapes do not match the worker.py:416-455 layout")
        return q, f, s, seg, im, vm, tk

    def __call__(self, *args, **kwargs):
        return self.forward(*args, **kwargs)

    @torch.no_grad()
    def forward(self, input_txt, input_imgs, image_loc, token_type_ids=None, attention_mask=None,
                image_attention_mask=None, co_attention_mask=None, task_ids=None,
                output_all_encoded_layers=False, output_all_attention_masks=False,
                compute_pretraining_heads=False, select: Optional[int] = None, debug_taps: bool = False, slot: int = 0):
        """Positional signature and 10-tuple of worker.py:286-289.

        ``vision_prediction`` / ``linguisic_prediction`` (the pre-training heads, elements 5 and 7, never read
        by the worker) are computed only with ``compute_pretraining_heads=True`` and are ``None`` otherwise;
        ``attn_data_list`` (element 9, never read by the worker) is the list of the 24 layers' attention probabilities in
        execution order -- ``[B, heads, L, L]`` for a text / image layer, a ``(text->image [B, heads, T, V], image->text
        [B, heads, V, T])`` tuple for a connection layer -- when ``output_all_attention_masks`` AND ``self.return_attention``
        are set, else ``[]``.  ``slot`` selects one of 16 independent workspaces: calls on different slots may be in flight
        concurrently on different CUDA streams.
        """
        if self._handle is None:
            if torch.is_tensor(input_txt) and input_txt.is_cuda:
                self.cuda(input_txt.device.index)
            else:
                raise L.VilbertB200Error("call model.cuda(i) first (worker.py:536); there is no CPU path")
        lib = L.load()
        device = torch.device("cuda", self._device)
        if select is None:
            select = L.OUT_ALL if compute_pretraining_heads else L.OUT_TASK_HEADS
        q, f, s, seg, im, vm, tk = self._prep(input_txt, input_imgs, image_loc, token_type_ids, attention_mask,
                                              image_attention_mask, task_ids, device)
        B, Tin = q.shape
        V = f.shape[1]
        inp = L.Inputs(B, Tin, V, q.data_ptr(), f.data_ptr(), s.data_ptr(), seg.data_ptr(), im.data_ptr(),
                       vm.data_ptr(), None, tk.data_ptr())
        want_attn = bool(output_all_attention_masks and self.return_attention)
        outs, o, select = self._alloc_outputs(B, Tin, V, select, debug_taps, want_attn, device)
        with torch.cuda.device(device):
            stream = torch.cuda.current_stream(device).cuda_stream
            L.check(lib.vb200_forward_slot(self._handle, C.byref(inp), C.byref(o), select, slot, C.c_void_p(stream)), self._handle)
        return self._result(outs, B, Tin, V, debug_taps)

    # ------------------------------------------------------------------ shared output plumbing
    def attention_layout(self, B, Tin, V):
        """[(heads, Lq, Lk, kind, float_offset)] of the flat attention buffer + its size (vb200_attention_layout)."""
        lib = L.load()
        n = C.c_int32()
        total = C.c_int64()
        L.check(lib.vb200_attention_layout(self._handle, B, Tin, V, 0, C.byref(n), None, None, C.byref(total)), self._handle)
        dims = (C.c_int32 * (4 * n.value))()
        offs = (C.c_int64 * n.value)()
        L.check(lib.vb200_attention_layout(self._handle, B, Tin, V, n.value, C.byref(n), dims, offs, C.byref(total)), self._handle)
        return [(dims[4 * i], dims[4 * i + 1], dims[4 * i + 2], dims[4 * i + 3], offs[i]) for i in range(n.value)], total.value

    def _alloc_outputs(self, B, Tin, V, select, debug_taps, want_attn, device):
        T = Tin + (1 if self._dims["task_specific_tokens"] else 0)
        outs = {k: torch.empty(shape, dtype=torch.float32, device=device)
                for k, shape in self._out_shapes(B, T, V, select).items()}
        if debug_taps:
            outs["sequence_output_t"] = torch.empty(B, T, self._dims["hidden_size"], dtype=torch.float32, device=device)
            outs["sequence_output_v"] = torch.empty(B, V, self._dims["v_hidden_size"], dtype=torch.float32, device=device)
            outs["pooled_output"] = torch.empty(B, self._dims["bi_hidden_size"], dtype=torch.float32, device=device)
        if want_attn:
            _, total = self.attention_layout(B, Tin, V)
            outs["attention_probs"] = torch.empty(total, dtype=torch.float32, device=device)
            select |= L.OUT_ATTENTION
        o = L.Outputs()
        for k, t in outs.items():
            setattr(o, k, t.data_ptr())
        return outs, o, select

    def _result(self, outs, B, Tin, V, debug_taps):
        g = outs.get
        attn = []
        if "attention_probs" in outs:
            flat = outs["attention_probs"]
            layout, _ = self.attention_layout(B, Tin, V)
            pending = None
            for heads, lq, lk, kind, off in layout:
                t = flat[off:off + B * heads * lq * lk].view(B, heads, lq, lk)
                if kind == 2:
                    pending = t
                elif kind == 3:
                    attn.append((pending, t))
                else:
                    attn.append(t)
        result = (g("vil_prediction"), g("vil_prediction_gqa"), g("vil_logit"), g("vil_binary_prediction"),
                  g("vil_tri_prediction"), g("vision_prediction"), g("vision_logit"), g("linguisic_prediction"),
                  g("linguisic_logit"), attn)
        if debug_taps:
            return result, {k: outs[k] for k in ("sequence_output_t", "sequence_output_v", "pooled_output")}
        return result

    # ------------------------------------------------------------------ detector output in, logits out (worker.py:388-458)
    @torch.no_grad()
    def forward_regions(self, question, segment_ids, input_mask, task_tokens, box_features, boxes, image_wh, num_boxes=None,
                        select: Optional[int] = None, output_all_attention_masks=False, slot: int = 0, return_spatials=True):
        """``custom_prediction``'s tensor construction fused into the forward: ``box_features [B, n, F]`` (what the detector
        returned, no global row), pixel ``boxes [B, n, 4]``, ``image_wh [B, 2]`` -> the 10-tuple (and the ``spatials``
        tensor ``[B, n+1, 5]`` the reference would have built: the grounding decode reads it, worker.py:379)."""
        if self._handle is None:
            raise L.VilbertB200Error("call model.cuda(i) first (worker.py:536); there is no CPU path")
        lib = L.load()
        device = torch.device("cuda", self._device)

        def dev(t, dtype):
            t = torch.as_tensor(t)
            return t.to(device=device, dtype=dtype, non_blocking=True).contiguous()
        q, seg, im = dev(question, torch.int64), dev(segment_ids, torch.int64), dev(input_mask, torch.int64)
        B, Tin = q.shape
        tk = dev(task_tokens, torch.int64).reshape(B, -1)[:, :1].contiguous()
        bf, bx, wh = dev(box_features, torch.float32), dev(boxes, torch.float32), dev(image_wh, torch.float32)
        n = bf.shape[1]
        if tuple(bf.shape) != (B, n, self._dims["v_feature_size"]) or tuple(bx.shape) != (B, n, 4) or tuple(wh.shape) != (B, 2) \
                or tuple(seg.shape) != (B, Tin) or tuple(im.shape) != (B, Tin):
            raise ValueError("forward_regions: box_features [B,n,F], boxes [B,n,4], image_wh [B,2], text [B,Tin] expected")
        nb = dev(num_boxes, torch.int32) if num_boxes is not None else None
        sp = torch.empty(B, n + 1, 5, dtype=torch.float32, device=device) if return_spatials else None
        if select is None:
            select = L.OUT_TASK_HEADS
        inp = L.RegionInputs(B, Tin, n, q.data_ptr(), seg.data_ptr(), im.data_ptr(), tk.data_ptr(), bf.data_ptr(), bx.data_ptr(),
                             wh.data_ptr(), nb.data_ptr() if nb is not None else None, sp.data_ptr() if sp is not None else None)
        want_attn = bool(output_all_attention_masks and self.return_attention)
        outs, o, select = self._alloc_outputs(B, Tin, n + 1, select, False, want_attn, device)
        with torch.cuda.device(device):
            stream = torch.cuda.current_stream(device).cuda_stream
            L.check(lib.vb200_forward_regions(self._handle, C.byref(inp), C.byref(o), select, slot, C.c_void_p(stream)), self._handle)
        return self._result(outs, B, Tin, n + 1, False), sp

    # ------------------------------------------------------------------ retrieval reuse (SURVEY.md section 8e)
    @torch.no_grad()
    def encode_text(self, question, segment_ids, input_mask, task_tokens):
        """Everything ahead of the first connection layer that depends on the caption alone (embeddings + text layers T0..),
        once per caption.  Returns an opaque state for ``forward_cached``."""
        lib = L.load()
        device = torch.device("cuda", self._device)
        q = question.to(device=device, dtype=torch.int64).contiguous()
        n, Tin = q.shape
        seg = segment_ids.to(device=device, dtype=torch.int64).contiguous()
        im = input_mask.to(device=device, dtype=torch.int64).contiguous()
        tk = task_tokens.to(device=device, dtype=torch.int64).reshape(n, -1)[:, :1].contiguous()
        T = Tin + (1 if self._dims["task_specific_tokens"] else 0)
        H, S = self._dims["hidden_size"], self._dims["operand_width_factor"]
        st = dict(kind="text", n=n, Tin=Tin, f32=torch.empty(n, T, H, dtype=torch.float32, device=device),
                  h16=torch.empty(n, T, H * S, dtype=torch.int16, device=device),
                  mask=torch.empty(n, T, dtype=torch.float32, device=device))
        with torch.cuda.device(device):
            stream = torch.cuda.current_stream(device).cuda_stream
            L.check(lib.vb200_encode_text(self._handle, n, Tin, q.data_ptr(), seg.data_ptr(), im.data_ptr(), tk.data_ptr(),
                                          st["f32"].data_ptr(), st["h16"].data_ptr(), st["mask"].data_ptr(), C.c_void_p(stream)),
                    self._handle)
        return st

    @torch.no_grad()
    def encode_image(self, features, spatials, image_mask):
        """The image-side prefix (image embedding, plus image layers scheduled ahead of the first connection layer), once per image."""
        lib = L.load()
        device = torch.device("cuda", self._device)
        f = features.to(device=device, dtype=torch.float32).contiguous()
        n, V = f.shape[0], f.shape[1]
        s = spatials.to(device=device, dtype=torch.float32).contiguous()
        vm = image_mask.to(device=device, dtype=torch.uint8).contiguous()
        Hv, S = self._dims["v_hidden_size"], self._dims["operand_width_factor"]
        st = dict(kind="image", n=n, V=V, f32=torch.empty(n, V, Hv, dtype=torch.float32, device=device),
                  h16=torch.empty(n, V, Hv * S, dtype=torch.int16, device=device),
                  mask=torch.empty(n, V, dtype=torch.float32, device=device))
        with torch.cuda.device(device):
            stream = torch.cuda.current_stream(device).cuda_stream
            L.check(lib.vb200_encode_image(self._handle, n, V, f.data_ptr(), s.data_ptr(), vm.data_ptr(), st["f32"].data_ptr(),
                                           st["h16"].data_ptr(), st["mask"].data_ptr(), C.c_void_p(stream)), self._handle)
        return st

    @torch.no_grad()
    def forward_cached(self, text_state, text_index, image_state, image_index, select: int = L.OUT_VIL_LOGIT, slot: int = 0):
        """Pair b = (caption text_index[b], image image_index[b]) from cached states: the connection layers onwards.  Results are
        bit-identical to the full forward of the same pairs."""
        lib = L.load()
        device = torch.device("cuda", self._device)
        ti = text_index.to(device=device, dtype=torch.int32).contiguous()
        vi = image_index.to(device=device, dtype=torch.int32).contiguous()
        B = ti.numel()
        if vi.numel() != B:
            raise ValueError("text_index and image_index must have the same length")
        Tin, V = text_state["Tin"], image_state["V"]
        outs, o, select = self._alloc_outputs(B, Tin, V, select, False, False, device)
        with torch.cuda.device(device):
            stream = torch.cuda.current_stream(device).cuda_stream
            L.check(lib.vb200_forward_cached(self._handle, B, Tin, V, ti.data_ptr(), text_state["n"], text_state["f32"].data_ptr(),
                                             text_state["h16"].data_ptr(), text_state["mask"].data_ptr(), vi.data_ptr(),
                                             image_state["n"], image_state["f32"].data_ptr(), image_state["h16"].data_ptr(),
                                             image_state["mask"].data_ptr(), C.byref(o), select, slot, C.c_void_p(stream)),
                    self._handle)
        return self._result(outs, B, Tin, V, False)

    # ------------------------------------------------------------------ host-buffer entry (bench e2e, serving)
    def forward_host(self, question, features, spatials, segment_ids, input_mask, image_mask, task_tokens,
                     out: Dict[str, torch.Tensor], select: int = L.OUT_VIL_PREDICTION, slot: int = 0, synchronize: bool = True):
        """vb200_forward_host[_slot]: HOST (ideally pinned) tensors in, HOST tensors out; H2D + forward + D2H (+ stream sync).
        With ``synchronize=False`` the call returns after enqueueing on the current stream; synchronise that stream before
        reading ``out`` or re-using the input buffers."""
        lib = L.load()
        B, Tin = question.shape
        V = features.shape[1]
        inp = L.Inputs(B, Tin, V, question.data_ptr(), features.data_ptr(), spatials.data_ptr(),
                       segment_ids.data_ptr(), input_mask.data_ptr(), image_mask.data_ptr(), None,
                       task_tokens.data_ptr())
        o = L.Outputs()
        for k, t in out.items():
            setattr(o, k, t.data_ptr())
        device = torch.device("cuda", self._device)
        with torch.cuda.device(device):
            stream = torch.cuda.current_stream(device).cuda_stream
            L.check(lib.vb200_forward_host_slot(self._handle, C.byref(inp), C.byref(o), select, slot, 1 if synchronize else 0,
                                                C.c_void_p(stream)), self._handle)
        return out
