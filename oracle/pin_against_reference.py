"""Pin oracle/hv_oracle.py against the reference's OWN Python modules and write tests/golden/.

Run in the build container only (needs /root/reference):

    python oracle/pin_against_reference.py            # check + (re)write tests/golden/*.pt

What is the real reference here: src/models/{unet_3d,unet_3d_blocks,resnet,transformer_3d,
attention,motion_module,mutual_self_attention,pose_guider}.py, the 2-D reference ("writer") UNet
src/models/{unet_2d_condition,unet_2d_blocks,transformer_2d}.py with the write hook and reader.update(writer), src/cameractrl/{pose_adaptor,
motion_module}.py, src/pipelines/context.py, src/dataset/dance_image_h_v_camera.py
(Camera, ray_condition) and scripts/pose2vid.py's get_relative_pose logic -- imported
unmodified from /root/reference.

What is NOT: ``diffusers==0.24.0`` (environment.yml:87) is not installed and there is no
network.  The few diffusers symbols those modules import are provided by the stand-ins below
(written from the published 0.24.0 algorithm, independently of oracle/hv_oracle.py's classes).
So this script pins (a) the oracle's restatement of every reference-owned file bit-for-bit,
and (b) that two independent restatements of the diffusers primitives agree; it cannot pin
the diffusers primitives against diffusers itself ("parity unpinned" for those, DESIGN.md).
"""
from __future__ import annotations

import os
import sys
import types
from collections import OrderedDict

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

REF = "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLD = os.path.join(ROOT, "tests", "golden")

# ------------------------------------------------------------------------------------------
# stand-ins for the diffusers 0.24.0 symbols the reference imports
# ------------------------------------------------------------------------------------------


class _Cfg(dict):
    __getattr__ = dict.__getitem__


def register_to_config(init):
    import functools
    import inspect

    @functools.wraps(init)
    def wrapper(self, *a, **kw):
        sig = inspect.signature(init)
        bound = sig.bind(self, *a, **kw)
        bound.apply_defaults()
        cfg = {k: v for k, v in bound.arguments.items() if k != "self"}
        object.__setattr__(self, "_cfg", _Cfg(cfg))
        init(self, *a, **kw)

    return wrapper


class ConfigMixin:
    @property
    def config(self):
        return self._cfg


class ModelMixin(nn.Module):
    @property
    def dtype(self):
        return next(self.parameters()).dtype

    @property
    def device(self):
        return next(self.parameters()).device


class BaseOutput:
    pass


class _Log:
    def get_logger(self, *_):
        import logging

        return logging.getLogger("ref")


class AttnProcessor2_0:
    def __call__(self, attn, hidden_states, encoder_hidden_states=None, attention_mask=None, **_):
        assert attention_mask is None
        ctx = hidden_states if encoder_hidden_states is None else encoder_hidden_states
        b, l, _c = hidden_states.shape
        q = attn.to_q(hidden_states)
        k = attn.to_k(ctx)
        v = attn.to_v(ctx)
        hd = q.shape[-1] // attn.heads
        q = q.view(b, -1, attn.heads, hd).transpose(1, 2)
        k = k.view(b, -1, attn.heads, hd).transpose(1, 2)
        v = v.view(b, -1, attn.heads, hd).transpose(1, 2)
        o = F.scaled_dot_product_attention(q, k, v, attn_mask=None, dropout_p=0.0, is_causal=False)
        o = o.transpose(1, 2).reshape(b, -1, attn.heads * hd).to(q.dtype)
        o = attn.to_out[1](attn.to_out[0](o))
        return o / attn.rescale_output_factor


class AttnProcessor(AttnProcessor2_0):
    pass


class DAttention(nn.Module):
    def __init__(self, query_dim, cross_attention_dim=None, heads=8, dim_head=64, dropout=0.0, bias=False,
                 upcast_attention=False, upcast_softmax=False, cross_attention_norm=None, added_kv_proj_dim=None,
                 norm_num_groups=None, out_bias=True, scale_qk=True, only_cross_attention=False,
                 rescale_output_factor=1.0, residual_connection=False, processor=None, **_):
        super().__init__()
        inner = dim_head * heads
        cdim = cross_attention_dim if cross_attention_dim is not None else query_dim
        self.heads = heads
        self.scale = dim_head ** -0.5
        self.rescale_output_factor = rescale_output_factor
        self.to_q = nn.Linear(query_dim, inner, bias=bias)
        self.to_k = nn.Linear(cdim, inner, bias=bias)
        self.to_v = nn.Linear(cdim, inner, bias=bias)
        self.to_out = nn.ModuleList([nn.Linear(inner, query_dim, bias=out_bias), nn.Dropout(dropout)])
        self.processor = processor or AttnProcessor2_0()

    def set_processor(self, p):
        self.processor = p

    def forward(self, hidden_states, encoder_hidden_states=None, attention_mask=None, **kw):
        return self.processor(self, hidden_states, encoder_hidden_states=encoder_hidden_states,
                              attention_mask=attention_mask, **kw)


class DGEGLU(nn.Module):
    def __init__(self, a, b):
        super().__init__()
        self.proj = nn.Linear(a, b * 2)

    def forward(self, x):
        x, gate = self.proj(x).chunk(2, dim=-1)
        return x * F.gelu(gate)


class DFeedForward(nn.Module):
    def __init__(self, dim, dim_out=None, mult=4, dropout=0.0, activation_fn="geglu", final_dropout=False):
        super().__init__()
        assert activation_fn == "geglu"
        inner = int(dim * mult)
        self.net = nn.ModuleList([DGEGLU(dim, inner), nn.Dropout(dropout), nn.Linear(inner, dim_out or dim)])

    def forward(self, x, scale=1.0):
        for m in self.net:
            x = m(x)
        return x


class Timesteps(nn.Module):
    def __init__(self, num_channels, flip_sin_to_cos, downscale_freq_shift):
        super().__init__()
        self.n, self.flip, self.shift = num_channels, flip_sin_to_cos, downscale_freq_shift

    def forward(self, timesteps):
        import math

        half = self.n // 2
        exponent = -math.log(10000) * torch.arange(0, half, dtype=torch.float32, device=timesteps.device)
        exponent = exponent / (half - self.shift)
        emb = timesteps[:, None].float() * torch.exp(exponent)[None, :]
        emb = torch.cat([torch.sin(emb), torch.cos(emb)], dim=-1)
        if self.flip:
            emb = torch.cat([emb[:, half:], emb[:, :half]], dim=-1)
        return emb


class DTimestepEmbedding(nn.Module):
    def __init__(self, in_channels, time_embed_dim, act_fn="silu", **_):
        super().__init__()
        self.linear_1 = nn.Linear(in_channels, time_embed_dim)
        self.act = nn.SiLU()
        self.linear_2 = nn.Linear(time_embed_dim, time_embed_dim)

    def forward(self, x, condition=None):
        return self.linear_2(self.act(self.linear_1(x)))


# ---- diffusers 0.24.0 2-D primitives the reference ("writer") UNet imports: resnet.py ResnetBlock2D / Downsample2D /
# Upsample2D and the LoRA-compatible layers (plain layers that ignore the lora ``scale`` argument when no LoRA is loaded)
class LoRACompatibleConv(nn.Conv2d):
    def forward(self, x, scale=1.0):
        return super().forward(x)


class LoRACompatibleLinear(nn.Linear):
    def forward(self, x, scale=1.0):
        return super().forward(x)


class DResnetBlock2D(nn.Module):
    def __init__(self, *, in_channels, out_channels=None, conv_shortcut=False, dropout=0.0, temb_channels=512, groups=32, groups_out=None,
                 pre_norm=True, eps=1e-6, non_linearity="swish", skip_time_act=False, time_embedding_norm="default", kernel=None,
                 output_scale_factor=1.0, use_in_shortcut=None, up=False, down=False, **_):
        super().__init__()
        assert time_embedding_norm == "default" and not up and not down and kernel is None
        out_channels = out_channels or in_channels
        self.output_scale_factor = output_scale_factor
        self.norm1 = nn.GroupNorm(groups, in_channels, eps=eps, affine=True)
        self.conv1 = LoRACompatibleConv(in_channels, out_channels, 3, stride=1, padding=1)
        self.time_emb_proj = LoRACompatibleLinear(temb_channels, out_channels) if temb_channels is not None else None
        self.norm2 = nn.GroupNorm(groups_out or groups, out_channels, eps=eps, affine=True)
        self.dropout = nn.Dropout(dropout)
        self.conv2 = LoRACompatibleConv(out_channels, out_channels, 3, stride=1, padding=1)
        self.nonlinearity = nn.SiLU()
        use_sc = in_channels != out_channels if use_in_shortcut is None else use_in_shortcut
        self.conv_shortcut = LoRACompatibleConv(in_channels, out_channels, 1, stride=1, padding=0) if use_sc else None

    def forward(self, input_tensor, temb, scale=1.0):
        h = self.conv1(self.nonlinearity(self.norm1(input_tensor)))
        if self.time_emb_proj is not None:
            h = h + self.time_emb_proj(self.nonlinearity(temb))[:, :, None, None]
        h = self.conv2(self.dropout(self.nonlinearity(self.norm2(h))))
        if self.conv_shortcut is not None:
            input_tensor = self.conv_shortcut(input_tensor)
        return (input_tensor + h) / self.output_scale_factor


class DDownsample2D(nn.Module):
    def __init__(self, channels, use_conv=False, out_channels=None, padding=1, name="conv"):
        super().__init__()
        assert use_conv and name in ("op", "conv")
        self.conv = LoRACompatibleConv(channels, out_channels or channels, 3, stride=2, padding=padding)   # name "op" -> attribute `conv`

    def forward(self, x, scale=1.0):
        return self.conv(x)


class DUpsample2D(nn.Module):
    def __init__(self, channels, use_conv=False, use_conv_transpose=False, out_channels=None, name="conv"):
        super().__init__()
        assert use_conv and not use_conv_transpose
        self.conv = LoRACompatibleConv(channels, out_channels or channels, 3, padding=1)

    def forward(self, x, output_size=None, scale=1.0):
        x = F.interpolate(x, scale_factor=2.0, mode="nearest") if output_size is None else F.interpolate(x, size=output_size, mode="nearest")
        return self.conv(x)


def install_stubs_2d():
    """Extra stand-ins needed to import src/models/{unet_2d_condition,unet_2d_blocks,transformer_2d}.py."""
    anyc = type("Any2", (nn.Module,), {})

    def mod(name, **attrs):
        m = sys.modules.get(name) or types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    mod("diffusers.loaders", UNet2DConditionLoadersMixin=type("UNet2DConditionLoadersMixin", (), {}))
    mod("diffusers.models.attention_processor", ADDED_KV_ATTENTION_PROCESSORS=(), CROSS_ATTENTION_PROCESSORS=(), AttnAddedKVProcessor=anyc)
    mod("diffusers.models.embeddings", GaussianFourierProjection=anyc, ImageHintTimeEmbedding=anyc, ImageProjection=anyc, ImageTimeEmbedding=anyc,
        PositionNet=anyc, TextImageProjection=anyc, TextImageTimeEmbedding=anyc, TextTimeEmbedding=anyc, CaptionProjection=anyc)
    mod("diffusers.utils", deprecate=lambda *a, **k: None, scale_lora_layers=lambda *a, **k: None, unscale_lora_layers=lambda *a, **k: None,
        is_torch_version=lambda op, v: True)
    mod("diffusers.utils.torch_utils", apply_freeu=lambda *a, **k: a)
    mod("diffusers.models.dual_transformer_2d", DualTransformer2DModel=anyc)
    mod("diffusers.models.resnet", Downsample2D=DDownsample2D, ResnetBlock2D=DResnetBlock2D, Upsample2D=DUpsample2D)
    mod("diffusers.models.lora", LoRACompatibleConv=LoRACompatibleConv, LoRACompatibleLinear=LoRACompatibleLinear)
    mod("diffusers.models.normalization", AdaLayerNormSingle=anyc)


def install_stubs():
    def mod(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    anyc = type("Any", (nn.Module,), {})
    mod("diffusers")
    mod("diffusers.configuration_utils", ConfigMixin=ConfigMixin, register_to_config=register_to_config)
    mod("diffusers.models", ModelMixin=ModelMixin)
    mod("diffusers.models.modeling_utils", ModelMixin=ModelMixin)
    mod("diffusers.models.attention_processor", AttentionProcessor=object, Attention=DAttention,
        AttnProcessor=AttnProcessor, SpatialNorm=anyc)
    mod("diffusers.models.attention", AdaLayerNorm=anyc, Attention=DAttention, FeedForward=DFeedForward)
    mod("diffusers.models.embeddings", TimestepEmbedding=DTimestepEmbedding, Timesteps=Timesteps,
        SinusoidalPositionalEmbedding=anyc)
    mod("diffusers.models.activations", get_activation=lambda n: nn.SiLU())
    mod("diffusers.models.normalization", AdaGroupNorm=anyc)
    mod("diffusers.models.lora", LoRALinearLayer=anyc)
    mod("diffusers.utils", SAFETENSORS_WEIGHTS_NAME="x.safetensors", WEIGHTS_NAME="x.bin", BaseOutput=BaseOutput,
        logging=_Log(), USE_PEFT_BACKEND=False)
    mod("diffusers.utils.import_utils", is_xformers_available=lambda: False)
    mod("decord", VideoReader=object)
    sys.path.insert(0, REF)


# ------------------------------------------------------------------------------------------


def maxdiff(a, b):
    return float((a.double() - b.double()).abs().max())


def main():
    sys.path.insert(0, ROOT)
    install_stubs()
    import contextlib
    import io

    from oracle import hv_oracle as O

    from src.models.unet_3d import UNet3DConditionModel as RefUNet
    from src.models.pose_guider import PoseGuider as RefPG
    from src.cameractrl.pose_adaptor import CameraPoseEncoder as RefCam
    from src.models.mutual_self_attention import ReferenceAttentionControl
    from src.pipelines.context import uniform as ref_uniform

    torch.manual_seed(0)
    os.makedirs(GOLD, exist_ok=True)
    report = OrderedDict()

    mm_kwargs = dict(num_attention_heads=8, num_transformer_block=1,
                     attention_block_types=["Temporal_Self", "Temporal_Self"], temporal_position_encoding=True,
                     temporal_position_encoding_max_len=32, temporal_attention_dim_div=1)

    def build_pair(chs, motion, xdim=768):
        ref = RefUNet(in_channels=4, out_channels=4, block_out_channels=chs, cross_attention_dim=xdim,
                      attention_head_dim=8, use_inflated_groupnorm=motion, use_motion_module=motion,
                      motion_module_resolutions=(1, 2, 4, 8), motion_module_mid_block=motion,
                      motion_module_type="Vanilla" if motion else None, motion_module_kwargs=mm_kwargs if motion else {},
                      unet_use_cross_frame_attention=False, unet_use_temporal_attention=False).eval()
        ora = O.UNet3DConditionModel(block_out_channels=chs, cross_attention_dim=xdim, use_motion_module=motion,
                                     use_inflated_groupnorm=motion).eval()
        O.synthetic_init(ora, seed=7)
        sd = ora.state_dict()
        missing, unexpected = ref.load_state_dict(sd, strict=False)
        # time_proj has no params; every key must match exactly
        assert not missing and not unexpected, (missing[:5], unexpected[:5])
        assert list(ref.state_dict().keys()) == list(sd.keys()) or set(ref.state_dict()) == set(sd)
        return ref, ora

    def run_ref(ref, *a, **kw):
        with contextlib.redirect_stdout(io.StringIO()), torch.no_grad():  # reference print()s in forward
            return ref(*a, **kw)

    # ---- 1. narrow UNet (fast; used as CPU golden) with motion modules, F=3 -----------------
    chs = (32, 64, 128, 128)
    ref, ora = build_pair(chs, True, xdim=64)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(2, 4, 3, 16, 16, generator=g)
    ehs = torch.randn(2, 1, 64, generator=g)
    pose = torch.randn(2, 32, 3, 16, 16, generator=g) * 0.5
    t = torch.tensor(721)
    y_ref = run_ref(ref, x, t, ehs, pose_cond_fea=pose, return_dict=False)[0]
    with torch.no_grad():
        y_ora = ora(x, t, ehs, pose_cond_fea=pose)[0]
    report["unet_narrow_motion"] = maxdiff(y_ref, y_ora)
    torch.save(dict(chs=chs, xdim=64, seed=7, x=x, ehs=ehs, pose=pose, t=721, y=y_ref), os.path.join(GOLD, "unet_narrow.pt"))

    # ---- 2. reference-attention read hook (CFG on and off) through the REAL ReferenceAttentionControl
    shapes = O.bank_shapes(ora, 16, 16)
    banks = [torch.randn(2, l, c, generator=g) for (l, c) in shapes]
    for cfg in (True, False):
        ctl = ReferenceAttentionControl(ref, do_classifier_free_guidance=cfg, mode="read", batch_size=1, fusion_blocks="full")
        from src.models.mutual_self_attention import torch_dfs
        from src.models.attention import TemporalBasicTransformerBlock as RefTB
        rmods = sorted([m for m in torch_dfs(ref) if isinstance(m, RefTB)], key=lambda m: -m.norm1.normalized_shape[0])
        assert [m.norm1.normalized_shape[0] for m in rmods] == [c for _, c in shapes]
        for m, bk in zip(rmods, banks):
            m.bank = [bk.clone()]
        y_ref_b = run_ref(ref, x, t, ehs, pose_cond_fea=pose, return_dict=False)[0]
        O.set_reference_banks(ora, banks, cfg=cfg)
        with torch.no_grad():
            y_ora_b = ora(x, t, ehs, pose_cond_fea=pose)[0]
        report[f"unet_narrow_bank_cfg{int(cfg)}"] = maxdiff(y_ref_b, y_ora_b)
        # un-hook the reference for the next round
        for m in rmods:
            m.forward = m._original_inner_forward
            m.bank = []
        O.set_reference_banks(ora, None)
        if cfg:
            torch.save(dict(banks=banks, y=y_ref_b), os.path.join(GOLD, "unet_narrow_bank.pt"))
            # the bank order must be: reader order == DFS(down, up, mid) stable-sorted by -dim
            names = {id(m): n for n, m in ref.named_modules()}
            report["bank_order"] = [names[id(m)] for m in rmods]

    # ---- 3. config-1 style UNet: no motion module, plain nn.GroupNorm, F=1 -------------------
    ref1, ora1 = build_pair(chs, False, xdim=64)
    x1 = torch.randn(2, 4, 1, 16, 16, generator=g)
    y_ref1 = run_ref(ref1, x1, t, ehs, pose_cond_fea=pose[:, :, :1], return_dict=False)[0]
    with torch.no_grad():
        y_ora1 = ora1(x1, t, ehs, pose_cond_fea=pose[:, :, :1])[0]
    report["unet_narrow_image"] = maxdiff(y_ref1, y_ora1)
    del ref1, ora1

    # ---- 4. full-width UNet (SD1.5 sizes), tiny spatial extent, F=2 -------------------------
    if os.environ.get("PIN_FULL", "1") == "1":
        reff, oraf = build_pair((320, 640, 1280, 1280), True, xdim=768)
        xf = torch.randn(2, 4, 2, 8, 8, generator=g)
        ehsf = torch.randn(2, 1, 768, generator=g)
        posef = torch.randn(2, 320, 2, 8, 8, generator=g) * 0.5
        y_reff = run_ref(reff, xf, torch.tensor(999), ehsf, pose_cond_fea=posef, return_dict=False)[0]
        with torch.no_grad():
            y_oraf = oraf(xf, torch.tensor(999), ehsf, pose_cond_fea=posef)[0]
        report["unet_full_width"] = maxdiff(y_reff, y_oraf)
        n_params = sum(p.numel() for p in oraf.parameters())
        report["unet_full_params"] = n_params
        torch.save(dict(seed=7, x=xf, ehs=ehsf, pose=posef, t=999, y=y_reff), os.path.join(GOLD, "unet_full_tiny.pt"))
        del reff, oraf

    # ---- 4b. reference ("writer") UNet2D + write hook + update() into the reader --------------------------------
    install_stubs_2d()
    from src.models.unet_2d_condition import UNet2DConditionModel as RefUNet2D

    def build_pair_2d(chs, xdim):
        with contextlib.redirect_stdout(io.StringIO()):
            ref2 = RefUNet2D(in_channels=4, out_channels=4, block_out_channels=chs, cross_attention_dim=xdim, attention_head_dim=8).eval()
        ora2 = O.synthetic_init(O.UNet2DConditionModel(block_out_channels=chs, cross_attention_dim=xdim).eval(), seed=17)
        missing, unexpected = ref2.load_state_dict(ora2.state_dict(), strict=False)
        assert not missing and not unexpected, (missing[:5], unexpected[:5])
        return ref2, ora2

    def ref_write(ref2, lat, ehs2):
        w = ReferenceAttentionControl(ref2, do_classifier_free_guidance=True, mode="write", batch_size=1, fusion_blocks="full")
        with torch.no_grad():
            hid = ref2(lat, torch.zeros((), dtype=torch.long), encoder_hidden_states=ehs2, return_dict=False)[0]
        from src.models.attention import BasicTransformerBlock as RefBTB
        blocks = sorted([m for m in torch_dfs_ref(ref2) if isinstance(m, RefBTB)], key=lambda m: -m.norm1.normalized_shape[0])
        return w, hid, [b.bank[0].clone() for b in blocks]

    from src.models.mutual_self_attention import torch_dfs as torch_dfs_ref

    ref2, ora2 = build_pair_2d((64, 128, 256, 256), 64)
    lat = torch.randn(1, 4, 16, 16, generator=g).repeat(2, 1, 1, 1)
    ehs2 = torch.cat([torch.zeros(1, 1, 64), torch.randn(1, 1, 64, generator=g)])
    writer, hid_ref, banks_ref = ref_write(ref2, lat, ehs2)
    O.set_reference_write(ora2)
    with torch.no_grad():
        hid_ora = ora2(lat, torch.tensor(0), ehs2)[0]
    banks_ora = O.written_banks(ora2)
    report["unet2d_writer_hidden"] = maxdiff(hid_ref, hid_ora)
    report["unet2d_writer_banks"] = max(maxdiff(a, b) for a, b in zip(banks_ref, banks_ora))
    report["unet2d_writer_bank_shapes"] = [list(b.shape) for b in banks_ref]
    assert len(banks_ref) == len(banks_ora) == 16
    # writer -> reader: reference update() chain vs oracle set_reference_banks(written_banks)
    ref3, ora3 = build_pair((64, 128, 256, 256), True, xdim=64)
    reader = ReferenceAttentionControl(ref3, do_classifier_free_guidance=True, mode="read", batch_size=1, fusion_blocks="full")
    reader.update(writer, dtype=torch.float32)
    x3 = torch.randn(2, 4, 3, 16, 16, generator=g)
    y3_ref = run_ref(ref3, x3, torch.tensor(519), ehs2, return_dict=False)[0]
    O.set_reference_banks(ora3, banks_ora, cfg=True)
    with torch.no_grad():
        y3_ora = ora3(x3, torch.tensor(519), ehs2)[0]
    report["unet2d_writer_to_reader_chain"] = maxdiff(y3_ref, y3_ora)
    # the 16 banks in full would take the file past 1 MB: keep a fixed, seeded quarter of each bank's tokens (both CFG halves)
    bank_rows = [torch.randperm(b.shape[1], generator=torch.Generator().manual_seed(i))[: max(1, b.shape[1] // 4)].sort().values
                 for i, b in enumerate(banks_ref)]
    torch.save(dict(seed=17, lat=lat, ehs=ehs2, hidden=hid_ref, bank_shapes=[tuple(b.shape) for b in banks_ref], bank_rows=bank_rows,
                    bank_samples=[b[:, r].clone() for b, r in zip(banks_ref, bank_rows)], seed3=7, x3=x3, t3=519, y3=y3_ref),
               os.path.join(GOLD, "unet2d_writer_narrow.pt"))
    reader.clear()
    writer.clear()
    del ref2, ora2, ref3, ora3
    if os.environ.get("PIN_FULL", "1") == "1":
        ref2, ora2 = build_pair_2d((320, 640, 1280, 1280), 768)
        latf = torch.randn(1, 4, 8, 8, generator=g).repeat(2, 1, 1, 1)
        ehs2f = torch.cat([torch.zeros(1, 1, 768), torch.randn(1, 1, 768, generator=g)])
        writer, hid_ref, banks_ref = ref_write(ref2, latf, ehs2f)
        O.set_reference_write(ora2)
        with torch.no_grad():
            hid_ora = ora2(latf, torch.tensor(0), ehs2f)[0]
        report["unet2d_writer_full_width_hidden"] = maxdiff(hid_ref, hid_ora)
        report["unet2d_writer_full_width_banks"] = max(maxdiff(a, b) for a, b in zip(banks_ref, O.written_banks(ora2)))
        report["unet2d_writer_full_params"] = sum(p.numel() for p in ora2.parameters())
        writer.clear()
        del ref2, ora2

    # ---- 5. PoseGuider -----------------------------------------------------------------------
    rpg = RefPG(320, block_out_channels=(16, 32, 96, 256)).eval()
    opg = O.synthetic_init(O.PoseGuider(320, 3, (16, 32, 96, 256)).eval(), seed=11)
    rpg.load_state_dict(opg.state_dict(), strict=True)
    img = torch.rand(1, 3, 2, 64, 48, generator=g)
    with torch.no_grad():
        a, b = rpg(img), opg(img)
    report["pose_guider"] = maxdiff(a, b)
    torch.save(dict(seed=11, x=img, y=a), os.path.join(GOLD, "pose_guider.pt"))

    # ---- 6. CameraPoseEncoder ------------------------------------------------------------------
    cam_kw = dict(downscale_factor=8, channels=[320], nums_rb=2, cin=384, ksize=1, sk=True, use_conv=False,
                  compression_factor=1, temporal_attention_nhead=8, attention_block_types=["Temporal_Self"],
                  temporal_position_encoding=True, temporal_position_encoding_max_len=24)
    rcam = RefCam(**cam_kw).eval()
    ocam = O.synthetic_init(O.CameraPoseEncoder().eval(), seed=13)
    rcam.load_state_dict(ocam.state_dict(), strict=True)
    pl = torch.randn(1, 6, 3, 64, 48, generator=g)
    with torch.no_grad():
        a, b = rcam(pl)[0], ocam(pl)[0]
    report["camera_encoder"] = maxdiff(a, b)
    torch.save(dict(seed=13, x=pl, y=a), os.path.join(GOLD, "camera_encoder.pt"))

    # ---- 7. context windows ------------------------------------------------------------------
    for nf in (24, 48, 87):
        r = list(ref_uniform(0, 25, nf, 24, 1, 4))
        o = O.uniform_windows(0, nf, 24, 1, 4)
        assert r == o, (nf, r, o)
    report["context_windows_48"] = [[w[0], w[-1]] for w in O.uniform_windows(0, 48, 24, 1, 4)]

    # ---- 8. Camera + ray_condition (Plucker) on a shipped trajectory ----------------------------
    import zipfile

    sys.modules.setdefault("src.dataset.visualization_utils", types.ModuleType("vz"))
    vz = sys.modules["src.dataset.visualization_utils"]
    for n in ("CameraPoseVisualizer", "visualize_camera_pose", "to_image", "pca_visualize"):
        setattr(vz, n, None)
    from src.dataset.dance_image_h_v_camera import Camera, ray_condition

    z = zipfile.ZipFile(os.path.join(REF, "data/test_set/camera_test_set.zip"))
    name = sorted(n for n in z.namelist() if n.endswith(".txt"))[0]
    rows = [[float(v) for v in ln.split()] for ln in z.read(name).decode().strip().splitlines()][:9]
    img_size = (48, 64)
    cams = [Camera(r, "test", img_size) for r in rows]
    tgt = list(range(1, 9))
    sel = [cams[0]] + [cams[i] for i in tgt]
    K = np.asarray([[c.fx * img_size[0], c.fy * img_size[1], c.cx * img_size[0], c.cy * img_size[1]] for c in sel[1:]], dtype=np.float32)
    abs2rel = np.eye(4) @ sel[0].w2c_mat
    poses = np.array([np.eye(4)] + [abs2rel @ c.c2w_mat for c in sel[1:]], dtype=np.float32)[1:]
    ref_pl = ray_condition(torch.as_tensor(K)[None], torch.as_tensor(poses)[None], img_size[1], img_size[0], device="cpu")[0]
    ref_pl = ref_pl.permute(0, 3, 1, 2).contiguous().unsqueeze(0)
    ora_pl = O.plucker_embedding(rows, 0, tgt, img_size)
    report["plucker"] = maxdiff(ref_pl, ora_pl)
    torch.save(dict(rows=rows, img_size=img_size, y=ref_pl.half()), os.path.join(GOLD, "plucker.pt"))

    # ---- 9. DDIM known answers (no reference implementation on disk: self-consistency pins) ----
    sch = O.DDIM()
    ts = sch.set_timesteps(25)
    report["ddim_timesteps_head_tail"] = [int(ts[0]), int(ts[1]), int(ts[-1])]
    report["ddim_alpha_bar_999"] = float(sch.alphas_cumprod[999])

    for k, v in report.items():
        print(f"{k}: {v}")
    bad = [k for k, v in report.items() if isinstance(v, float) and k not in ("ddim_alpha_bar_999",) and v > 1e-4]
    assert not bad, bad
    import json

    with open(os.path.join(GOLD, "pin_report.json"), "w") as f:
        json.dump(report, f, indent=1)
    print("PIN OK")


if __name__ == "__main__":
    main()
