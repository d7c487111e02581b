"""Pin humanvid_b200/pipeline.py's HOST loop against the reference's OWN pipeline code (row a15 of SURVEY 8a and the pipeline half of the boundary).

Run with a checkout of the reference tree (pin_against_reference.REF):

    python oracle/pin_pipeline_against_reference.py        # check + (re)write tests/golden/pipeline_pin_report.json and
                                                            # tests/golden/pipeline_reference_outputs.pt

and without it, against the reference pipeline's outputs stored by that run (on the CPU: the pipelines use a GPU when they see one):

    CUDA_VISIBLE_DEVICES= python oracle/pin_pipeline_against_reference.py --against-golden

What is compared: ``src/pipelines/pipeline_pose2vid_long.py::Pose2VideoPipeline.__call__`` and ``src/pipelines/pipeline_pose2img.py::
Pose2ImagePipeline.__call__``, imported UNMODIFIED from /root/reference, against ``humanvid_b200.pipeline.Pose2VideoPipeline / Pose2ImagePipeline``
-- both driving the SAME module objects (the reference's own UNet3D / UNet2D / PoseGuider / CameraPoseEncoder classes with the reference's own
ReferenceAttentionControl, a stand-in VAE and CLIP encoder, this package's DDIM scheduler) on CPU in fp32.  With identical modules every
difference would come from the pipeline itself: CLIP / VAE preprocessing, latent preparation, the writer forward and ``reader.update(writer)``,
context windows, accumulation and ``counter``, the CFG mix (incl. the reference's quirk that ``/ counter`` only happens under CFG), the scheduler
calls, latent interpolation and the decode.  Expected and required: every difference is exactly 0.0 (one fp32 ulp for the batched VAE decode,
which changes the call pattern into the VAE on purpose).

``--against-golden`` repeats every case with this package's pipeline driving oracle/hv_oracle.py's restatement of the same modules (pinned
bit-for-bit to the reference's by pin_against_reference.py) under the oracle's bank hooks, and compares with a fixed, seeded sample of what
the reference's pipeline returned.

As in pin_against_reference.py the diffusers symbols the reference imports (``DiffusionPipeline``, ``VaeImageProcessor``, ``randn_tensor`` ...)
are stand-ins: diffusers 0.24.0 is not installed.  They are plumbing here (module registration, PIL -> tensor, ``torch.randn``); the loop under
test is the reference's own file.
"""
from __future__ import annotations

import contextlib
import io
import json
import os
import sys
import types
from collections import OrderedDict

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import pin_against_reference as P  # noqa: E402  (the stand-ins for the model-side diffusers symbols)

GOLD = os.path.join(ROOT, "tests", "golden")
GOLDEN_OUTPUTS = os.path.join(GOLD, "pipeline_reference_outputs.pt")
CHS, XDIM = (32, 64, 64, 64), 32
H = W = 64


# ------------------------------------------------------------------------------------------ pipeline-side stand-ins
class DiffusionPipeline:
    """register_modules / progress_bar / to: what the reference pipelines use of diffusers' base class."""

    def register_modules(self, **kw):
        for k, v in kw.items():
            setattr(self, k, v)

    @contextlib.contextmanager
    def progress_bar(self, iterable=None, total=None):
        class _Bar:
            def update(self, *_):
                pass

        yield _Bar()

    def to(self, *a, **k):
        return self


class VaeImageProcessor:
    """diffusers.image_processor.VaeImageProcessor.preprocess for PIL input: RGB -> resize to a multiple of the VAE factor (lanczos)
    -> [0, 1] float32 NCHW -> [-1, 1] when do_normalize."""

    def __init__(self, do_resize=True, vae_scale_factor=8, resample="lanczos", do_normalize=True, do_binarize=False, do_convert_rgb=False,
                 do_convert_grayscale=False):
        self.do_resize, self.f, self.do_normalize, self.do_convert_rgb = do_resize, vae_scale_factor, do_normalize, do_convert_rgb
        assert resample == "lanczos" and not do_binarize and not do_convert_grayscale

    def preprocess(self, image, height=None, width=None):
        from PIL import Image

        images = image if isinstance(image, list) else [image]
        out = []
        for im in images:
            assert isinstance(im, Image.Image)
            if self.do_convert_rgb:
                im = im.convert("RGB")
            if self.do_resize:
                h = height if height is not None else im.height
                w = width if width is not None else im.width
                w, h = (x - x % self.f for x in (w, h))
                im = im.resize((w, h), resample=Image.LANCZOS)
            out.append(np.array(im).astype(np.float32) / 255.0)
        t = torch.from_numpy(np.stack(out, axis=0).transpose(0, 3, 1, 2))
        return 2.0 * t - 1.0 if self.do_normalize else t


def randn_tensor(shape, generator=None, device=None, dtype=None, layout=None):
    gdev = generator.device if generator is not None else device
    return torch.randn(shape, generator=generator, device=gdev, dtype=dtype).to(device)


def _config_getattr(self, name):
    """diffusers' ModelMixin.__getattr__: attributes that are not modules / parameters fall back to the registered config
    (the pipelines read ``denoising_unet.in_channels``, pipeline_pose2vid_long.py:409)."""
    try:
        return nn.Module.__getattr__(self, name)
    except AttributeError:
        cfg = self.__dict__.get("_cfg")
        if cfg is not None and name in cfg:
            return cfg[name]
        raise


def install_pipeline_stubs():
    P.install_stubs()
    P.install_stubs_2d()
    P.ModelMixin.__getattr__ = _config_getattr

    def mod(name, **attrs):
        m = sys.modules.get(name) or types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    sched = type("AnyScheduler", (), {})
    mod("diffusers", DiffusionPipeline=DiffusionPipeline)
    mod("diffusers.image_processor", VaeImageProcessor=VaeImageProcessor)
    mod("diffusers.schedulers", DDIMScheduler=sched, DPMSolverMultistepScheduler=sched, EulerAncestralDiscreteScheduler=sched,
        EulerDiscreteScheduler=sched, LMSDiscreteScheduler=sched, PNDMScheduler=sched)
    mod("diffusers.utils", deprecate=lambda *a, **k: None, is_accelerate_available=lambda: False, BaseOutput=P.BaseOutput, logging=P._Log())
    mod("diffusers.utils.torch_utils", randn_tensor=randn_tensor)


# ------------------------------------------------------------------------------------------ VAE / CLIP stand-ins (same objects for both pipelines)
class StubVAE(nn.Module):
    """Deterministic stand-in with the AutoencoderKL surface the pipelines touch (config.block_out_channels, encode().latent_dist.mean,
    decode().sample, dtype, device)."""

    def __init__(self):
        super().__init__()
        self.config = types.SimpleNamespace(block_out_channels=(1, 2, 3, 4))
        self.enc = nn.Conv2d(3, 4, 1)
        self.dec = nn.Conv2d(4, 3, 3, padding=1)
        self.decode_calls = []

    @property
    def dtype(self):
        return self.enc.weight.dtype

    @property
    def device(self):
        return self.enc.weight.device

    def encode(self, x):
        return types.SimpleNamespace(latent_dist=types.SimpleNamespace(mean=self.enc(F.avg_pool2d(x, 8))))

    def decode(self, z):
        self.decode_calls.append(int(z.shape[0]))
        return types.SimpleNamespace(sample=torch.tanh(self.dec(F.interpolate(z, scale_factor=8.0, mode="nearest"))))


class StubCLIP(nn.Module):
    def __init__(self, dim):
        super().__init__()
        self.proj = nn.Linear(3, dim)

    @property
    def dtype(self):
        return self.proj.weight.dtype

    def forward(self, pix):
        return types.SimpleNamespace(image_embeds=self.proj(pix.mean(dim=(2, 3))))


def maxdiff(a, b):
    a, b = torch.as_tensor(a), torch.as_tensor(b)
    assert a.shape == b.shape, (a.shape, b.shape)
    return float((a.double() - b.double()).abs().max())


def pipeline_inputs():
    """Reference image (not the target size: the resize paths are exercised), 12 pose images and the camera embedding."""
    from PIL import Image

    rng = np.random.RandomState(3)

    def pil(h=H, w=W):
        return Image.fromarray(rng.randint(0, 256, size=(h, w, 3), dtype=np.uint8))

    ref_image = pil(80, 72)
    poses = [pil() for _ in range(12)]
    camera = torch.randn(1, 6, 12, H, W, generator=torch.Generator().manual_seed(4))
    return ref_image, poses, camera


def output_sample(t, seed, n=1024):
    """A fixed, seeded sample of n values of a pipeline output: all of them would take the golden file past 1 MB."""
    idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(seed))[:n]
    return {"shape": tuple(t.shape), "idx": idx.int(), "values": t.reshape(-1)[idx].clone()}


def main(write=True):
    install_pipeline_stubs()
    from oracle import hv_oracle as O

    import humanvid_b200.pipeline as HP
    from humanvid_b200.scheduler import DDIMScheduler

    from src.cameractrl.pose_adaptor import CameraPoseEncoder as RefCam
    from src.models.mutual_self_attention import ReferenceAttentionControl as RefControl
    from src.models.pose_guider import PoseGuider as RefPG
    from src.models.unet_2d_condition import UNet2DConditionModel as RefUNet2D
    from src.models.unet_3d import UNet3DConditionModel as RefUNet3D
    import src.pipelines.utils as ref_utils
    from src.pipelines.pipeline_pose2img import Pose2ImagePipeline as RefImagePipe
    from src.pipelines.pipeline_pose2vid_long import Pose2VideoPipeline as RefVideoPipe

    torch.manual_seed(0)
    report = OrderedDict()
    chs, xdim = CHS, XDIM
    mmk = dict(num_attention_heads=8, num_transformer_block=1, attention_block_types=["Temporal_Self", "Temporal_Self"],
               temporal_position_encoding=True, temporal_position_encoding_max_len=32, temporal_attention_dim_div=1)

    def quiet(fn, *a, **k):
        with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
            return fn(*a, **k)

    def unet3d(motion):
        ref = quiet(RefUNet3D, in_channels=4, out_channels=4, block_out_channels=chs, cross_attention_dim=xdim, attention_head_dim=8,
                    use_inflated_groupnorm=motion, use_motion_module=motion, motion_module_resolutions=(1, 2, 4, 8), motion_module_mid_block=motion,
                    motion_module_type="Vanilla" if motion else None, motion_module_kwargs=mmk if motion else {},
                    unet_use_cross_frame_attention=False, unet_use_temporal_attention=False).eval()
        ora = O.synthetic_init(O.UNet3DConditionModel(block_out_channels=chs, cross_attention_dim=xdim, use_motion_module=motion,
                                                      use_inflated_groupnorm=motion).eval(), seed=7)
        ref.load_state_dict(ora.state_dict(), strict=True)
        return ref

    unet2d = quiet(RefUNet2D, in_channels=4, out_channels=4, block_out_channels=chs, cross_attention_dim=xdim, attention_head_dim=8).eval()
    unet2d.load_state_dict(O.synthetic_init(O.UNet2DConditionModel(block_out_channels=chs, cross_attention_dim=xdim).eval(), seed=17).state_dict(), strict=True)
    pg = RefPG(chs[0], block_out_channels=(16, 32, 64, 128)).eval()
    pg.load_state_dict(O.synthetic_init(O.PoseGuider(chs[0], 3, (16, 32, 64, 128)).eval(), seed=11).state_dict(), strict=True)
    cam = RefCam(downscale_factor=8, channels=[chs[0]], nums_rb=2, cin=384, ksize=1, sk=True, use_conv=False, compression_factor=1,
                 temporal_attention_nhead=8, attention_block_types=["Temporal_Self"], temporal_position_encoding=True,
                 temporal_position_encoding_max_len=24).eval()
    cam.load_state_dict(O.synthetic_init(O.CameraPoseEncoder(channels=(chs[0],), heads=8).eval(), seed=13).state_dict(), strict=True)
    vae, clip = StubVAE().eval(), StubCLIP(xdim).eval()
    for p in list(vae.parameters()) + list(clip.parameters()):
        p.requires_grad_(False)
    golden = {"vae": vae.state_dict(), "clip": clip.state_dict(), "outputs": {}}
    ref_image, poses, camera = pipeline_inputs()

    def pipes(denoising):
        r = RefVideoPipe(vae=vae, image_encoder=clip, reference_unet=unet2d, denoising_unet=denoising, pose_guider=pg, camera_pose_encoder=cam,
                         scheduler=DDIMScheduler())
        n = HP.Pose2VideoPipeline(vae=vae, image_encoder=clip, reference_unet=unet2d, denoising_unet=denoising, pose_guider=pg, camera_pose_encoder=cam,
                                  scheduler=DDIMScheduler())
        n.reference_control_cls = (RefControl, RefControl)      # INTEGRATION.md: the reference's own control classes around its PyTorch UNets
        n.vae_decode_batch = 1                                   # the reference's call pattern (one frame per decode)
        return r, n

    den = unet3d(True)
    rpipe, npipe = pipes(den)

    def both(tag, n_frames, guidance, steps=2, decode_batch=1, **kw):
        npipe.vae_decode_batch = decode_batch
        a = quiet(rpipe, ref_image, poses[:n_frames], camera[:, :, :n_frames], W, H, n_frames, steps, guidance, generator=torch.Generator().manual_seed(9),
                  context_frames=8, context_stride=1, context_overlap=2, **kw).videos
        b = quiet(npipe, ref_image, poses[:n_frames], camera[:, :, :n_frames], W, H, n_frames, steps, guidance, generator=torch.Generator().manual_seed(9),
                  context_frames=8, context_stride=1, context_overlap=2, **kw).videos
        assert torch.isfinite(a).all() and float(a.std()) > 1e-3
        report[tag] = maxdiff(a, b)
        golden["outputs"][tag] = output_sample(a, len(golden["outputs"]))
        return a, b

    # the windows of the multi-window cases (context.py): 12 frames, 8 per window, overlap 2 -> two windows, frames covered once or twice
    report["windows_12_8_2"] = [list(map(int, w)) for w in HP.uniform(0, 2, 12, 8, 1, 2)]
    both("video_cfg_two_windows", 12, 3.5)
    both("video_no_cfg_two_windows_sum_quirk", 12, 1.0)           # pipeline_pose2vid_long.py:551-555: no `/ counter` without CFG
    both("video_cfg_single_window", 8, 3.5)
    both("video_cfg_three_steps", 12, 2.0, steps=3)
    a, b = both("video_cfg_decode_batch_8", 12, 3.5, decode_batch=8)   # batched VAE decode (SURVEY 8f-4): same frames, other call pattern
    report["decode_calls_reference_then_native"] = [vae.decode_calls[-14:-2], vae.decode_calls[-2:]]
    ref_utils.set_tensor_interpolation_method(True)
    HP.set_tensor_interpolation_method(True)
    both("video_cfg_interpolation_factor_2_slerp", 8, 3.5, interpolation_factor=2)
    ref_utils.set_tensor_interpolation_method(False)
    HP.set_tensor_interpolation_method(False)
    both("video_cfg_interpolation_factor_3_linear", 8, 3.5, interpolation_factor=3)
    # a per-step callback: the reference's window-batching loop shadows `i`, so its callback sees (num_context_batches - 1) // order as the step
    # index (documented deviation: ours passes the true step index); the latents handed over must agree
    seen_r, seen_n = [], []
    both("video_cfg_with_callback", 12, 3.5, callback=lambda i, t, lat: seen_r.append((int(i), int(t), lat.clone())), callback_steps=1)
    seen_r, seen_split = seen_r[: len(seen_r) // 2], seen_r[len(seen_r) // 2:]
    report["callback_step_index_reference"], report["callback_step_index_native"] = [s[0] for s in seen_r], [s[0] for s in seen_split]
    report["callback_latents"] = max(maxdiff(x[2], y[2]) for x, y in zip(seen_r, seen_split)) if seen_r and len(seen_r) == len(seen_split) else None
    report["callback_timesteps_equal"] = [s[1] for s in seen_r] == [s[1] for s in seen_split]
    golden["callback_latents"] = [s[2] for s in seen_r]

    # ---- Pose2ImagePipeline (config 1 plumbing): no motion modules, one frame ------------------------------------------------------------
    den1 = unet3d(False)
    rimg = RefImagePipe(vae=vae, image_encoder=clip, reference_unet=unet2d, denoising_unet=den1, pose_guider=pg, camera_pose_encoder=cam,
                        scheduler=DDIMScheduler())
    nimg = HP.Pose2ImagePipeline(vae=vae, image_encoder=clip, reference_unet=unet2d, denoising_unet=den1, pose_guider=pg, camera_pose_encoder=cam,
                                 scheduler=DDIMScheduler())
    nimg.reference_control_cls = (RefControl, RefControl)
    nimg.vae_decode_batch = 1
    cam4 = camera[:, :, 0]
    for tag, guidance in (("image_cfg", 3.5), ("image_no_cfg", 1.0)):
        a = quiet(rimg, ref_image, poses[0], cam4, W, H, 2, guidance, generator=torch.Generator().manual_seed(5)).images
        b = quiet(nimg, ref_image, poses[0], cam4, W, H, 2, guidance, generator=torch.Generator().manual_seed(5)).images
        assert torch.isfinite(a).all() and float(a.std()) > 1e-3
        report[tag] = maxdiff(a, b)
        golden["outputs"][tag] = output_sample(a, len(golden["outputs"]))

    # the batched decode feeds the VAE 8 frames per call instead of 1: same arithmetic per frame, but a CPU convolution may block a batch of 8
    # differently from a batch of 1 -- one fp32 ulp is allowed there, everything else must be bit-identical
    tol = {"video_cfg_decode_batch_8": 1e-6}
    bad = {k: v for k, v in report.items() if isinstance(v, float) and v > tol.get(k, 0.0)}
    for k, v in report.items():
        print(f"{k:48s} {v}")
    if write:
        os.makedirs(GOLD, exist_ok=True)
        json.dump(report, open(os.path.join(GOLD, "pipeline_pin_report.json"), "w"), indent=1)
        torch.save(golden, GOLDEN_OUTPUTS)
    if bad:
        raise SystemExit(f"pipeline differs from the reference: {bad}")
    return report


class OracleControl:
    """ReferenceAttentionControl(fusion_blocks="full") of mutual_self_attention.py for oracle/hv_oracle.py's UNets, through the write and
    read hooks the oracle restates; update() hands the banks over in ``dtype`` like the reference's."""

    def __init__(self, unet, do_classifier_free_guidance=False, mode="read", **_):
        from oracle import hv_oracle as O

        self.O, self.unet, self.mode, self.cfg = O, unet, mode, do_classifier_free_guidance
        if mode == "write":
            O.set_reference_write(unet)

    def update(self, writer, dtype=torch.float16):
        self.O.set_reference_banks(self.unet, [b.clone().to(dtype) for b in self.O.written_banks(writer.unet)], cfg=self.cfg)

    def clear(self):
        if self.mode == "read":
            self.O.set_reference_banks(self.unet, None)
        else:
            self.O.set_reference_write(self.unet)


def against_golden():
    """Every case of main() with this package's pipeline on the oracle's modules, against the stored outputs of the reference's pipeline.
    On the CPU the golden file was made on the two agree exactly (the batched decode to one ulp).  Another CPU's kernels differ in the
    last bits, and the no-CFG case, which sums overlapping windows, amplifies that to ~1e-4 on the [0, 1] frames; a pipeline fault
    (averaging there, a wrong window, CFG mix or scheduler call) moves them by orders of magnitude more than TOL."""
    from oracle import hv_oracle as O

    import humanvid_b200.pipeline as HP
    from humanvid_b200.scheduler import DDIMScheduler

    TOL = 1e-3
    gold = torch.load(GOLDEN_OUTPUTS, weights_only=False)
    report = OrderedDict()

    def unet3d(motion):
        return O.synthetic_init(O.UNet3DConditionModel(block_out_channels=CHS, cross_attention_dim=XDIM, use_motion_module=motion,
                                                       use_inflated_groupnorm=motion).eval(), seed=7)

    unet2d = O.synthetic_init(O.UNet2DConditionModel(block_out_channels=CHS, cross_attention_dim=XDIM).eval(), seed=17)
    pg = O.synthetic_init(O.PoseGuider(CHS[0], 3, (16, 32, 64, 128)).eval(), seed=11)
    cam = O.synthetic_init(O.CameraPoseEncoder(channels=(CHS[0],), heads=8).eval(), seed=13)
    vae, clip = StubVAE().eval(), StubCLIP(XDIM).eval()
    vae.load_state_dict(gold["vae"])
    clip.load_state_dict(gold["clip"])
    for p in list(vae.parameters()) + list(clip.parameters()):
        p.requires_grad_(False)
    ref_image, poses, camera = pipeline_inputs()

    def compare(tag, out):
        g = gold["outputs"][tag]
        assert tuple(out.shape) == g["shape"], (tag, tuple(out.shape), g["shape"])
        report[tag] = maxdiff(out.reshape(-1)[g["idx"].long()], g["values"])

    with torch.no_grad():
        npipe = HP.Pose2VideoPipeline(vae=vae, image_encoder=clip, reference_unet=unet2d, denoising_unet=unet3d(True), pose_guider=pg,
                                      camera_pose_encoder=cam, scheduler=DDIMScheduler())
        npipe.reference_control_cls = (OracleControl, OracleControl)

        def video(tag, n_frames, guidance, steps=2, decode_batch=1, **kw):
            npipe.vae_decode_batch = decode_batch
            compare(tag, npipe(ref_image, poses[:n_frames], camera[:, :, :n_frames], W, H, n_frames, steps, guidance,
                               generator=torch.Generator().manual_seed(9), context_frames=8, context_stride=1, context_overlap=2, **kw).videos)

        video("video_cfg_two_windows", 12, 3.5)
        video("video_no_cfg_two_windows_sum_quirk", 12, 1.0)
        video("video_cfg_single_window", 8, 3.5)
        video("video_cfg_three_steps", 12, 2.0, steps=3)
        video("video_cfg_decode_batch_8", 12, 3.5, decode_batch=8)
        report["decode_calls_native"] = vae.decode_calls[-2:]
        HP.set_tensor_interpolation_method(True)
        video("video_cfg_interpolation_factor_2_slerp", 8, 3.5, interpolation_factor=2)
        HP.set_tensor_interpolation_method(False)
        video("video_cfg_interpolation_factor_3_linear", 8, 3.5, interpolation_factor=3)
        seen = []
        video("video_cfg_with_callback", 12, 3.5, callback=lambda i, t, lat: seen.append((int(i), lat.clone())), callback_steps=1)
        report["callback_step_index_native"] = [s[0] for s in seen]
        report["callback_latents"] = max(maxdiff(s[1], g) for s, g in zip(seen, gold["callback_latents"]))
        assert len(seen) == len(gold["callback_latents"])

        nimg = HP.Pose2ImagePipeline(vae=vae, image_encoder=clip, reference_unet=unet2d, denoising_unet=unet3d(False), pose_guider=pg,
                                     camera_pose_encoder=cam, scheduler=DDIMScheduler())
        nimg.reference_control_cls = (OracleControl, OracleControl)
        nimg.vae_decode_batch = 1
        for tag, guidance in (("image_cfg", 3.5), ("image_no_cfg", 1.0)):
            compare(tag, nimg(ref_image, poses[0], camera[:, :, 0], W, H, 2, guidance, generator=torch.Generator().manual_seed(5)).images)

    for k, v in report.items():
        print(f"{k:48s} {v}")
    bad = {k: v for k, v in report.items() if isinstance(v, float) and v > TOL}
    if bad or report["decode_calls_native"] != [8, 4] or report["callback_step_index_native"] != [0, 1]:
        raise SystemExit(f"pipeline differs from the reference's stored outputs: {bad}")
    print("against golden OK")


if __name__ == "__main__":
    if "--against-golden" in sys.argv:
        against_golden()
    else:
        main(write="--check" not in sys.argv)
