"""VTPModel — the drop-in boundary (SURVEY.md §8b): same Python surface, attribute names and state-dict keys as
the reference's vtp/models/vtp_hf/modeling_vtp.py:51-472, with every FLOP executed by the sm_100a kernels in
libvtp_b200.so (see engine.py).  There is no eager/PyTorch fallback: on a CUDA-less host the API methods raise.

Precision follows the caller's autocast context exactly like the reference does:
  torch.autocast("cuda", bfloat16) active  -> "bf16" mode (bf16 tensor-core GEMMs / attention)
  otherwise                               -> "fp32" mode (bf16x3-split GEMMs, fp32-accurate; what
                                             tools/test_reconstruction_hf.py:369-372 uses for the decoder)
`model.compute_mode = "bf16" | "fp32"` overrides the detection.

Small-batch serving (BASELINE config 5, batch 1..512): `model.enable_cuda_graphs()` captures each inference entry point
once per (input shape, dtype, precision mode) in a CUDA graph and replays it afterwards — a VTP-Large encode+decode is
~1 000 kernel launches, which at batch 1 costs more host time than device time.

Checkpoints: `from_pretrained(dir)` / `save_pretrained(dir)` read/write the reference's HF layout (config.json +
model.safetensors, keys unchanged).  The text tower needs no `attn_mask` buffer (causality is applied in-kernel), which
also removes the reference's uninitialised-buffer NaN after from_pretrained under transformers 5.x (SURVEY.md M8).
"""
from __future__ import annotations

import json
import math
import os
from typing import Dict, Optional, Sequence, Tuple, Union

import torch
from torch import nn

from . import engine as E
from . import lib
from .config import VTPConfig
from .rope import rope_periods

BF = torch.bfloat16


def _swiglu_hidden(dim: int, ratio: float, ffn_layer: str) -> int:
    """layers/block.py:176 + layers/ffn.py:71-72 (+ align variants encoders/vision_transformer.py:22-28)."""
    align = {"swiglu": 8, "swiglu32": 32, "swiglu64": 64, "swiglu128": 128}[ffn_layer]
    d = int(int(dim * ratio) * 2 / 3)
    return d + (-d % align)


def check_head_dims(c: VTPConfig) -> None:
    """The attention / RoPE kernels (forward and backward) address the packed [M, 3D] qkv buffer as H heads of 64
    columns (csrc/attention.cu: D = H * 64): every tower that runs must have embed_dim == 64 * num_heads, otherwise the
    kernels would read with the wrong stride.  The reference accepts other head sizes; this path does not."""
    towers = [("vision", c.vision_embed_dim, c.vision_num_heads)]
    if c.train_reconstruction:
        towers.append(("decoder", c.decoder_embed_dim, c.decoder_num_heads))
    if c.train_clip:
        towers.append(("text", c.text_embed_dim, c.text_num_heads))
    for name, dim, heads in towers:
        if heads <= 0 or dim != 64 * heads:
            raise NotImplementedError(f"{name} tower: embed_dim {dim} / num_heads {heads} gives head_dim != 64; the "
                                      "B200 attention kernels are specialised for head_dim == 64")


class _Holder(nn.Module):
    """Parameter container (no forward): gives the reference's module-path state-dict keys."""


def _param(*shape):
    return nn.Parameter(torch.empty(*shape))


def _linear_holder(n_out, n_in, bias=True):
    h = _Holder()
    h.weight = _param(n_out, n_in)
    if bias:
        h.bias = _param(n_out)
    return h


def _norm_holder(dim, ln: bool):
    h = _Holder()
    h.weight = _param(dim)
    if ln:
        h.bias = _param(dim)
    return h


def _vit_block_holder(dim, hidden, ln: bool):
    b = _Holder()
    b.norm1 = _norm_holder(dim, ln)
    b.attn = _Holder()
    b.attn.qkv = _linear_holder(3 * dim, dim)
    b.attn.proj = _linear_holder(dim, dim)
    b.norm2 = _norm_holder(dim, ln)
    b.mlp = _Holder()
    b.mlp.w1 = _linear_holder(hidden, dim)
    b.mlp.w2 = _linear_holder(hidden, dim)
    b.mlp.w3 = _linear_holder(dim, hidden)
    return b


class VTPPreTrainedModel(nn.Module):
    config_class = VTPConfig
    base_model_prefix = "vtp"


class VTPModel(VTPPreTrainedModel):
    def __init__(self, config: VTPConfig):
        super().__init__()
        self.config = config
        self.compute_mode: Optional[str] = None
        c = config
        for flag, what in ((c.vision_init_values, "vision LayerScale"), (c.decoder_init_values, "decoder LayerScale"),
                           (c.text_ls_init_value, "text LayerScale")):
            if flag is not None:
                raise NotImplementedError(f"{what} is not implemented by the B200 path (reference default is None)")
        if c.vision_use_qk_norm or c.decoder_use_qk_norm:
            raise NotImplementedError("qk-norm is not implemented by the B200 path (reference default is False)")
        check_head_dims(c)
        self._init_vision_components()
        if c.train_clip:
            self._init_text_components()
        self.reset_parameters()
        self._packs: Dict[Tuple[str, str], Tuple[int, E.TowerW]] = {}
        self._graphs_on = False          # see enable_cuda_graphs()
        self._graph_busy = False         # True while a graph is being warmed up / captured (the eager path runs)
        self._graphs: Dict[tuple, tuple] = {}

    # ------------------------------------------------------------------ CUDA graphs for the inference entry points
    def enable_cuda_graphs(self, on: bool = True):
        """Replay captured CUDA graphs for get_reconstruction_latents / get_latents_decoded_images /
        get_clip_image_feature / get_clip_text_feature (one graph per input shape, dtype and precision mode; dropped
        when the parameters change).  Results are identical to the eager launches: the same kernels in the same order."""
        self._graphs_on = bool(on)
        if not on:
            self._graphs = {}
        return self

    def _graphed(self, name: str, fn, x: torch.Tensor, *extra):
        """Run fn(x) through a captured graph: static input buffer <- x, replay, fresh copy of the static output."""
        if not x.is_cuda:
            raise lib.VtpError("VTPModel inputs must live on the CUDA device (no CPU path)")
        key = (name, tuple(x.shape), x.dtype, self._mode(), extra)
        ver = self._version()
        hit = self._graphs.get(key)
        if hit is None or hit[0] != ver:
            static_in = x.detach().clone()
            cur = torch.cuda.current_stream()
            side = torch.cuda.Stream()
            side.wait_stream(cur)
            self._graph_busy = True
            try:
                with torch.cuda.stream(side):    # warm-up: packs the weights, builds RoPE tables, sizes the allocator
                    for _ in range(2):
                        fn(static_in)
                cur.wait_stream(side)
                torch.cuda.synchronize()
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    static_out = fn(static_in)
            finally:
                self._graph_busy = False
            hit = (ver, graph, static_in, static_out)
            self._graphs[key] = hit
        _, graph, static_in, static_out = hit
        static_in.copy_(x)
        graph.replay()
        return static_out.clone()

    # ------------------------------------------------------------------ parameters (reference names)
    def _init_vision_components(self):
        c = self.config
        D = c.vision_embed_dim
        ln = c.vision_norm_layer != "rmsnorm"
        t = _Holder()
        t.cls_token = _param(1, 1, D)
        t.mask_token = _param(1, D)
        t.patch_embed = _Holder()
        t.patch_embed.proj = _Holder()
        t.patch_embed.proj.weight = _param(D, 3, c.vision_patch_size, c.vision_patch_size)
        t.patch_embed.proj.bias = _param(D)
        t.rope_embed = _Holder()
        t.rope_embed.register_buffer("periods", rope_periods(D // c.vision_num_heads), persistent=True)
        hs = _swiglu_hidden(D, c.vision_mlp_ratio, c.vision_ffn_layer)
        t.blocks = nn.ModuleList([_vit_block_holder(D, hs, ln) for _ in range(c.vision_depth)])
        t.norm = _norm_holder(D, ln)
        if c.vision_feature_bottleneck is not None and c.vision_feature_bottleneck != D:
            t.feature_bottleneck = _linear_holder(c.vision_feature_bottleneck, D, bias=False)
        t.embed_dim = D
        t.vit_feature_bottleneck = c.vision_feature_bottleneck or D
        self.trunk = t
        eff = t.vit_feature_bottleneck
        if c.train_clip:
            self.visual_proj = _linear_holder(c.text_embed_dim, D if c.vision_bottleneck_ae_only else eff, bias=False)
        else:
            self.visual_proj = None
        if c.train_reconstruction:
            Dd = c.decoder_embed_dim
            lnd = c.decoder_norm_layer != "rmsnorm"
            d = _Holder()
            d.proj_in = _Holder()
            d.proj_in.weight = _param(Dd, eff, 1, 1)
            d.proj_in.bias = _param(Dd)
            d.rope_embed = _Holder()
            d.rope_embed.register_buffer("periods", rope_periods(Dd // c.decoder_num_heads), persistent=True)
            hsd = _swiglu_hidden(Dd, 4.0, c.decoder_ffn_layer)
            d.blocks = nn.ModuleList([_vit_block_holder(Dd, hsd, lnd) for _ in range(c.decoder_depth)])
            d.norm = _norm_holder(Dd, lnd)
            d.proj_out = _Holder()
            d.proj_out.weight = _param(3 * 16 * 16, Dd, 1, 1)
            d.proj_out.bias = _param(3 * 16 * 16)
            self.pixel_decoder = d
        else:
            self.pixel_decoder = None

    def _init_text_components(self):
        c = self.config
        Dt = c.text_embed_dim
        if c.text_embed_cls or c.text_no_causal_mask or c.text_pool_type != "argmax" or c.text_proj_bias or \
                c.text_quick_gelu or c.text_proj_type != "linear":
            raise NotImplementedError("only the reference's default text tower (causal, argmax pool, GELU, linear "
                                      "projection without bias) is implemented by the B200 path")
        tt = _Holder()
        blocks = []
        for _ in range(c.text_depth):
            b = _Holder()
            b.ln_1 = _norm_holder(Dt, True)
            b.attn = _Holder()
            b.attn.in_proj_weight = _param(3 * Dt, Dt)
            b.attn.in_proj_bias = _param(3 * Dt)
            b.attn.out_proj = _linear_holder(Dt, Dt)
            b.ln_2 = _norm_holder(Dt, True)
            b.mlp = _Holder()
            b.mlp.c_fc = _linear_holder(int(Dt * c.text_mlp_ratio), Dt)
            b.mlp.c_proj = _linear_holder(Dt, int(Dt * c.text_mlp_ratio))
            blocks.append(b)
        tt.resblocks = nn.ModuleList(blocks)
        self.text_transformer = tt
        self.context_length = c.text_context_length
        self.vocab_size = c.text_vocab_size
        self.token_embedding = _Holder()
        self.token_embedding.weight = _param(c.text_vocab_size, Dt)
        self.positional_embedding = _param(c.text_context_length, Dt)
        self.ln_final = _norm_holder(Dt, True)
        self.text_projection = _param(Dt, Dt)
        self.text_pool_type = c.text_pool_type
        init_logit_scale = c.init_logit_scale or math.log(1 / 0.07)
        lshape = [1] if c.nonscalar_logit_scale else []
        self.logit_scale = nn.Parameter(torch.ones(lshape) * init_logit_scale)
        self.logit_bias = nn.Parameter(torch.ones(lshape) * c.init_logit_bias) if c.init_logit_bias is not None else None

    @torch.no_grad()
    def reset_parameters(self):
        """Same distributions as the reference's constructors + HF post_init (vision_transformer.py:43-55,181-187;
        embeddings.py:79-83; pixel_decoder.py:123-132; text_transformer.py:301-324; modeling_vtp.py:38-48).
        Parity tests copy a reference state dict instead of relying on RNG order."""
        c = self.config
        for name, p in self.named_parameters():
            leaf = name.rsplit(".", 1)[-1]
            if name in ("logit_scale", "logit_bias"):
                continue
            if name == "trunk.cls_token":
                nn.init.normal_(p, std=0.02)
            elif name == "trunk.mask_token":
                nn.init.zeros_(p)
            elif name.startswith("trunk.patch_embed.proj"):
                k = 1 / (3 * c.vision_patch_size ** 2)
                nn.init.uniform_(p, -math.sqrt(k), math.sqrt(k))
            elif name == "positional_embedding":
                nn.init.normal_(p, std=0.01)
            elif name == "token_embedding.weight":
                nn.init.normal_(p, std=0.02)
            elif name == "text_projection":
                nn.init.normal_(p, std=c.text_embed_dim ** -0.5)
            elif name.endswith("attn.in_proj_weight"):
                nn.init.normal_(p, std=c.text_embed_dim ** -0.5)
            elif leaf in ("bias", "in_proj_bias"):
                nn.init.zeros_(p)
            elif ("norm" in name or ".ln_" in name or name.startswith("ln_final")) and leaf == "weight":
                nn.init.ones_(p)
            elif leaf == "weight":
                nn.init.trunc_normal_(p, std=0.02)
            else:  # pragma: no cover
                raise RuntimeError(f"no init rule for {name}")

    # ------------------------------------------------------------------ HF-format checkpoints
    @classmethod
    def from_pretrained(cls, path: str, device: Optional[Union[str, torch.device]] = None,
                        torch_dtype: Optional[torch.dtype] = None, device_map: Optional[Union[str, torch.device]] = None, **kwargs):
        """HF checkpoint directory (config.json + model.safetensors, or the sharded `model.safetensors.index.json` layout).
        `torch_dtype` converts the stored parameters (compute precision still follows the caller's autocast context);
        `device_map` accepts a single device ("cuda", "cuda:0", torch.device) — sharding a model over devices is not
        supported.  Hub names and any other `PreTrainedModel.from_pretrained` argument raise instead of being ignored."""
        from safetensors.torch import load_file

        if kwargs:
            raise TypeError(f"VTPModel.from_pretrained: unsupported arguments {sorted(kwargs)} (local directory, torch_dtype, "
                            "device / device_map only)")
        if not os.path.isdir(path):
            raise FileNotFoundError(f"{path!r} is not a local checkpoint directory (hub names need network access)")
        if device_map is not None:
            if isinstance(device_map, dict) or device_map in ("auto", "balanced", "sequential"):
                raise NotImplementedError("device_map must name ONE device; model sharding is not supported")
            device = device_map if device is None else device
        with open(os.path.join(path, "config.json")) as f:
            cd = json.load(f)
        for k in ("architectures", "model_type", "transformers_version", "torch_dtype", "dtype"):
            cd.pop(k, None)
        model = cls(VTPConfig(**cd))
        index = os.path.join(path, "model.safetensors.index.json")
        if os.path.exists(index):          # sharded checkpoint: {"weight_map": {key: shard file}}
            with open(index) as f:
                shards = sorted(set(json.load(f)["weight_map"].values()))
            sd = {}
            for sh in shards:
                sd.update(load_file(os.path.join(path, sh)))
        else:
            sd = load_file(os.path.join(path, "model.safetensors"))
        missing, unexpected = model.load_state_dict(sd, strict=False)
        missing = [k for k in missing if not k.endswith("rope_embed.periods")]
        if missing or unexpected:
            raise RuntimeError(f"checkpoint mismatch: missing={missing[:5]} unexpected={unexpected[:5]}")
        if torch_dtype is not None:
            periods = {k: v.clone() for k, v in model.state_dict().items() if k.endswith("rope_embed.periods")}
            model = model.to(torch_dtype)
            model.load_state_dict(periods, strict=False)     # the bf16 RoPE periods buffer keeps its dtype
        return model.to(device) if device is not None else model

    def save_pretrained(self, path: str):
        from safetensors.torch import save_file

        os.makedirs(path, exist_ok=True)
        cd = {k: v for k, v in self.config.to_dict().items()}
        cd["model_type"] = "vtp"
        cd["architectures"] = ["VTPModel"]
        with open(os.path.join(path, "config.json"), "w") as f:
            json.dump(cd, f, indent=2, default=str)
        save_file({k: v.detach().cpu().contiguous() for k, v in self.state_dict().items()},
                  os.path.join(path, "model.safetensors"))

    def load_state_dict(self, state_dict, strict: bool = True, **kw):
        sd = {k: v for k, v in state_dict.items() if k != "attn_mask"}  # reference's non-persistent buffer
        out = super().load_state_dict(sd, strict=strict, **kw)
        self._packs = {}
        return out

    # ------------------------------------------------------------------ packing / mode
    def _mode(self) -> str:
        if self.compute_mode is not None:
            return self.compute_mode
        if torch.is_autocast_enabled("cuda") and torch.get_autocast_dtype("cuda") == BF:
            return "bf16"
        return "fp32"

    def _version(self):
        """Cache key of the packed weights / captured graphs: in-place version counters AND where the parameters live
        (`.to(device)`, `.half()` or `p.data = ...` do not bump `_version`).  Writers through `p.data.copy_()` must call
        `invalidate_packed_weights()`."""
        p0 = self.trunk.cls_token
        return (sum(p._version for p in self.parameters()), str(p0.device), p0.dtype, p0.data_ptr())

    def invalidate_packed_weights(self):
        self._packs = {}
        self._graphs = {}

    def _apply(self, fn, *args, **kwargs):     # .to() / .cuda() / .half(): packed copies and graphs point at the old storage
        out = super()._apply(fn, *args, **kwargs)
        if hasattr(self, "_packs"):
            self._packs, self._graphs = {}, {}
        return out

    def _pack(self, tower: str, mode: str) -> E.TowerW:
        ver = self._version()
        hit = self._packs.get((tower, mode))
        if hit is not None and hit[0] == ver:
            return hit[1]
        dev = self.trunk.cls_token.device
        if dev.type != "cuda":
            raise lib.VtpError("VTPModel runs only on a CUDA (sm_100a) device; move the model with .cuda() — there is "
                               "no CPU path")
        lib.check(lib.load().vtp_check_device(), "vtp_check_device")
        sd = {k: v for k, v in self.state_dict().items()}
        with torch.no_grad():
            if tower == "trunk":
                W = E.pack_trunk(sd, self.config, mode)
                if self.visual_proj is not None:
                    W.extra["visual_proj"] = E.pack_lin(sd["visual_proj.weight"], None, mode)
            elif tower == "decoder":
                W = E.pack_decoder(sd, self.config, mode)
            elif tower == "text":
                W = E.pack_text(sd, self.config, mode)
            else:  # pragma: no cover
                raise KeyError(tower)
        self._packs[(tower, mode)] = (ver, W)
        return W

    def _check_image(self, image: torch.Tensor):
        if image.dim() != 4 or image.shape[1] != 3:
            raise ValueError(f"expected image of shape (B, 3, H, W), got {tuple(image.shape)}")
        ps = self.config.vision_patch_size
        if image.shape[-1] % ps or image.shape[-2] % ps:
            raise ValueError(f"image size {tuple(image.shape[-2:])} is not a multiple of the patch size {ps}")
        if not image.is_cuda:
            raise lib.VtpError("VTPModel inputs must live on the CUDA device (no CPU path)")

    @torch.no_grad()
    def _trunk(self, image, use_bottleneck: bool, mode: str):
        self._check_image(image)
        W = self._pack("trunk", mode)
        x, meta = E.trunk_forward(W, image, mode)
        return E.trunk_outputs(W, x, meta, mode, use_bottleneck=use_bottleneck), meta, W

    # ------------------------------------------------------------------ public API (modeling_vtp.py:184-472)
    def get_last_layer_feature(self, image: torch.Tensor, use_bottleneck: bool = False) -> Dict[str, torch.Tensor]:
        out, _, _ = self._trunk(image, use_bottleneck, self._mode())
        return {"cls_token": out["x_norm_clstoken"], "patch_tokens": out["x_norm_patchtokens"]}

    @torch.no_grad()
    def get_intermediate_layers_feature(self, image, n: Union[int, Sequence[int]] = 1, reshape: bool = False,
                                        return_class_token: bool = False, norm: bool = True):
        """encoders/vision_transformer.py:266-318 (bottleneck bypassed, vision_transformer_bottleneck.py:81-98)."""
        self._check_image(image)
        mode = self._mode()
        W = self._pack("trunk", mode)
        depth = len(W.blocks)
        # the reference collects outputs while walking the blocks (vision_transformer.py:266-279): ascending block order
        # whatever the order of `n`, and every requested index must exist exactly once
        take = list(range(depth - n, depth)) if isinstance(n, int) else sorted(n)
        assert len(set(take)) == len(take) and all(0 <= i < depth for i in take), f"only {len(set(take))} / {len(take)} blocks found"
        taps = {i: None for i in take}
        _, meta = E.trunk_forward(W, image, mode, taps=taps)
        B, T, gh, gw = meta
        outs = []
        for i in take:
            x = taps[i]
            if norm:
                x = E.norm(x, B * T, W.D, W.norm_w, W.norm_b, W.eps, mode, want="f32")
            outs.append(x.view(B, T, W.D))
        cls_tokens = [o[:, 0] for o in outs]
        patches = [o[:, 1:] for o in outs]
        if reshape:
            patches = [p.reshape(B, gh, gw, -1).permute(0, 3, 1, 2).contiguous() for p in patches]
        if return_class_token:
            return tuple(zip(patches, cls_tokens))
        return tuple(patches)

    @torch.no_grad()
    def get_clip_image_feature(self, image: torch.Tensor, normalize: bool = True) -> torch.Tensor:
        if self.visual_proj is None:
            raise RuntimeError("CLIP not enabled. Set train_clip=True in config.")
        if self._graphs_on and image.is_cuda and not self._graph_busy:
            self._check_image(image)
            return self._graphed("clip_image", lambda t: self.get_clip_image_feature(t, normalize), image, normalize)
        mode = self._mode()
        out, meta, W = self._trunk(image, not self.config.vision_bottleneck_ae_only, mode)
        if self.config.vision_clip_feat == "cls":
            feat = out["x_norm_clstoken"]
        elif self.config.vision_clip_feat == "pooled":
            raise NotImplementedError("vision_clip_feat='pooled' is not implemented by the B200 path")
        else:
            raise ValueError(f"Invalid vision_clip_feat: {self.config.vision_clip_feat}")
        B = feat.shape[0]
        vp: E.Lin = W.extra["visual_proj"]
        act = BF if mode == "bf16" else torch.float32
        feat = feat.to(act).contiguous()  # strided cls rows -> dense [B, D] (cast == autocast's input cast)
        f = torch.empty((B, vp.N), dtype=act, device=feat.device)
        E.linear(E.operand(feat, B, vp.K, mode), vp, f, B, mode)
        return E.l2_normalize(f) if normalize else f

    @torch.no_grad()
    def get_clip_text_feature(self, text: torch.Tensor, normalize: bool = True) -> torch.Tensor:
        if not self.config.train_clip:
            raise RuntimeError("CLIP not enabled. Set train_clip=True in config.")
        if text.dtype != torch.int64 or text.dim() != 2 or text.shape[1] != self.config.text_context_length:
            raise ValueError(f"expected int64 token ids of shape (B, {self.config.text_context_length})")
        if self._graphs_on and text.is_cuda and not self._graph_busy:
            return self._graphed("clip_text", lambda t: self.get_clip_text_feature(t, normalize), text, normalize)
        mode = self._mode()
        W = self._pack("text", mode)
        f = E.text_forward(W, text, mode)
        return E.l2_normalize(f) if normalize else f

    @torch.no_grad()
    def get_clip_logits(self, image: torch.Tensor, text: torch.Tensor):
        fi = self.get_clip_image_feature(image, normalize=True)
        ft = self.get_clip_text_feature(text, normalize=True)
        mode = self._mode()
        Bi, Bt, Edim = fi.shape[0], ft.shape[0], fi.shape[1]
        # logit_scale.exp() * I @ T.T (+ bias)  (modeling_vtp.py:329-331): scale folded into the A operand
        scale = self.logit_scale.detach().exp().to(fi.dtype)
        a = (fi * scale).contiguous()
        logits = torch.empty((Bi, (Bt + 7) // 8 * 8), dtype=fi.dtype, device=fi.device)
        bt = ft
        if Bt % 8:
            bt = torch.zeros((logits.shape[1], Edim), dtype=ft.dtype, device=ft.device)
            bt[:Bt] = ft
        if mode == "bf16":
            lib.gemm(a, bt, logits, M=Bi, N=logits.shape[1], K=Edim)
        else:
            b3 = torch.empty((bt.shape[0], 3 * Edim), dtype=BF, device=ft.device)
            lib.split3(bt, b3, bt.shape[0], Edim, b_side=True)
            lib.gemm(E.operand(a, Bi, Edim, mode), b3, logits, M=Bi, N=logits.shape[1], K=3 * Edim, round_bf16=False)
        logits = logits[:, :Bt]
        if self.logit_bias is not None:
            logits = logits + self.logit_bias.detach().to(logits.dtype)
        return logits, logits.T

    def get_reconstruction_latents(self, image: torch.Tensor) -> torch.Tensor:
        if self._graphs_on and image.is_cuda and not self._graph_busy:
            self._check_image(image)
            return self._graphed("latents", self.get_reconstruction_latents, image)
        out, meta, _ = self._trunk(image, True, self._mode())
        _, _, gh, gw = meta
        pt = out["x_norm_patchtokens"]
        if pt.shape[1] != gh * gw:
            raise ValueError(f"Patch count mismatch: {pt.shape[1]} vs {gh * gw}")
        return E.latents_nchw(pt, gh, gw)

    @torch.no_grad()
    def get_latents_decoded_images(self, latents: torch.Tensor) -> torch.Tensor:
        if self.pixel_decoder is None:
            raise RuntimeError("Reconstruction not enabled. Set train_reconstruction=True in config.")
        if not latents.is_cuda:
            raise lib.VtpError("VTPModel inputs must live on the CUDA device (no CPU path)")
        if self._graphs_on and latents.is_cuda and not self._graph_busy:
            return self._graphed("decode", self.get_latents_decoded_images, latents)
        mode = self._mode()
        return E.decoder_forward(self._pack("decoder", mode), latents, mode)

    def forward(self, image: Optional[torch.Tensor] = None, text: Optional[torch.Tensor] = None,
                forward_type: str = "clip") -> Dict[str, torch.Tensor]:
        if forward_type == "clip":
            result = {}
            if image is not None:
                result["image_features"] = self.get_clip_image_feature(image, normalize=True)
            if text is not None:
                result["text_features"] = self.get_clip_text_feature(text, normalize=True)
            result["logit_scale"] = self.logit_scale.exp()
            if self.logit_bias is not None:
                result["logit_bias"] = self.logit_bias
            return result
        elif forward_type == "rec":
            if image is None:
                raise ValueError("image is required for reconstruction")
            latents = self.get_reconstruction_latents(image)
            return {"latents": latents, "reconstructed_image": self.get_latents_decoded_images(latents),
                    "target_image": image}
        elif forward_type == "feature":
            if image is None:
                raise ValueError("image is required for feature extraction")
            return self.get_last_layer_feature(image, use_bottleneck=True)
        raise ValueError(f"Invalid forward_type: {forward_type}")
