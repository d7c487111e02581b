"""Network-level parity on a B200: the native UNet3DConditionModel / PoseGuider / CameraPoseEncoder (through the C ABI)
against the oracle on identical weights and inputs, the committed golden vectors (generated from the reference's own
modules), and size-independent properties at the BASELINE config-2 shape.

Tolerances.  north_star: <= 1e-3 relative (fp16) per tensor vs the reference PyTorch path.  Per operator (tests/test_ops_gpu.py) and
per block on identical inputs (tests/test_ladder_gpu.py) that is what is asserted.  Through a whole network the fp16 storage roundings
of ~65 sequential tensors accumulate to ~1.5e-3 in ANY fp16 implementation (the reference's own fp16-eager path: 1.7e-3), so there:
  * err(native, fp32 oracle) <= err(fp16-eager oracle, fp32 oracle) + 1e-4   (native is no further from exact than the reference's deployment)
  * err(native, fp16-eager oracle) <= 2.5e-3
"""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden")

from conftest import report

if torch.cuda.is_available():
    import humanvid_b200 as hv
    from oracle import hv_oracle as O

MM_KW = dict(num_attention_heads=8, num_transformer_block=1, attention_block_types=["Temporal_Self", "Temporal_Self"],
             temporal_position_encoding=True, temporal_position_encoding_max_len=32, temporal_attention_dim_div=1)


def rel(a, b):
    a, b = a.float(), b.float()
    return float((a - b).norm() / (b.norm() + 1e-12))


def make_unet(chs, xdim, seed=7, motion=True):
    ora = O.UNet3DConditionModel(block_out_channels=chs, cross_attention_dim=xdim, use_motion_module=motion, use_inflated_groupnorm=motion).eval()
    O.synthetic_init(ora, seed=seed)
    ora = ora.half().float().cuda()  # weights exactly representable in fp16: native and oracle see the same numbers
    kw = dict(block_out_channels=chs, cross_attention_dim=xdim, unet_use_cross_frame_attention=False, unet_use_temporal_attention=False)
    if motion:
        kw.update(use_motion_module=True, use_inflated_groupnorm=True, motion_module_resolutions=(1, 2, 4, 8), motion_module_mid_block=True,
                  motion_module_type="Vanilla", motion_module_kwargs=MM_KW)
    nat = hv.UNet3DConditionModel(**kw)
    nat.load_state_dict(ora.state_dict())
    nat = nat.to("cuda", torch.float16)
    return ora, nat


def unet_inputs(B, F, h, w, c0, xdim, seed=1):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(B, 4, F, h, w, generator=g, device="cuda").half()
    ehs = torch.randn(B, 1, xdim, generator=g, device="cuda").half()
    ehs[: B // 2] = 0  # uncond half, like the pipeline
    pose = (torch.randn(B, c0, F, h, w, generator=g, device="cuda") * 0.5).half()
    return x, ehs, pose


@pytest.fixture(scope="module")
def narrow():
    return make_unet((64, 128, 256, 256), 64)


def run3(ora, nat, x, t, ehs, pose):
    with torch.no_grad():
        y32 = ora(x.float(), torch.tensor(t, device="cuda"), ehs.float(), pose_cond_fea=pose.float())[0]
        o16 = ora.half()
        y16 = o16(x, torch.tensor(t, device="cuda"), ehs, pose_cond_fea=pose)[0]
        ora.float()
        yn = nat(x, t, ehs, pose_cond_fea=pose, return_dict=False)[0]
    torch.cuda.synchronize()
    return y32, y16, yn


def test_unet_narrow_parity(narrow):
    ora, nat = narrow
    x, ehs, pose = unet_inputs(2, 5, 16, 16, 64, 64)
    y32, y16, yn = run3(ora, nat, x, 721, ehs, pose)
    e_ref, e_nat, e_pair = rel(y16, y32), rel(yn, y32), rel(yn, y16)
    report(f"narrow: fp16-eager vs fp32 {e_ref:.2e}; native vs fp32 {e_nat:.2e}; native vs fp16-eager {e_pair:.2e}")
    assert torch.isfinite(yn).all()
    assert e_nat <= e_ref + 1e-4
    assert e_pair <= 2.5e-3


def test_unet_narrow_reference_banks_and_cfg(narrow):
    ora, nat = narrow
    B, F = 2, 3
    x, ehs, pose = unet_inputs(B, F, 16, 16, 64, 64, seed=3)
    g = torch.Generator(device="cuda").manual_seed(5)
    banks = [torch.randn(B, l, c, generator=g, device="cuda").half() for (l, c) in O.bank_shapes(ora, 16, 16)]
    with torch.no_grad():
        y_plain = nat(x, 500, ehs, pose_cond_fea=pose, return_dict=False)[0].clone()
    ctl = hv.ReferenceAttentionControl(nat, do_classifier_free_guidance=True, mode="read", fusion_blocks="full")
    for blk, bk in zip(nat.reader_blocks(), banks):
        blk.bank = [bk]
    O.set_reference_banks(ora, [b.float() for b in banks], cfg=True)
    with torch.no_grad():
        y32 = ora(x.float(), torch.tensor(500, device="cuda"), ehs.float(), pose_cond_fea=pose.float())[0]
        yn = nat(x, 500, ehs, pose_cond_fea=pose, return_dict=False)[0].clone()
    O.set_reference_banks(ora, None)
    torch.cuda.synchronize()
    report(f"narrow + banks + CFG: native vs fp32 {rel(yn, y32):.2e}")
    assert rel(yn, y32) < 2.5e-3
    # CFG semantics: the uncond half never sees the bank -> bitwise equal to the plain forward; the cond half changes
    assert torch.equal(yn[:1], y_plain[:1])
    assert rel(yn[1:], y_plain[1:]) > 1e-2
    # without CFG every row reads the bank
    ctl2 = hv.ReferenceAttentionControl(nat, do_classifier_free_guidance=False, mode="read", fusion_blocks="full")
    for blk, bk in zip(nat.reader_blocks(), banks):
        blk.bank = [bk]
    O.set_reference_banks(ora, [b.float() for b in banks], cfg=False)
    with torch.no_grad():
        y32b = ora(x.float(), torch.tensor(500, device="cuda"), ehs.float(), pose_cond_fea=pose.float())[0]
        ynb = nat(x, 500, ehs, pose_cond_fea=pose, return_dict=False)[0]
    O.set_reference_banks(ora, None)
    ctl2.clear()
    assert rel(ynb, y32b) < 2.5e-3
    with torch.no_grad():
        y_again = nat(x, 500, ehs, pose_cond_fea=pose, return_dict=False)[0]
    assert torch.equal(y_again, y_plain)  # clear() restores plain self-attention, and the forward is deterministic


def test_unet_image_variant_no_motion_module():
    ora, nat = make_unet((64, 128, 256, 256), 64, motion=False)
    x, ehs, pose = unet_inputs(2, 1, 32, 32, 64, 64, seed=9)
    y32, y16, yn = run3(ora, nat, x, 999, ehs, pose)
    report(f"image variant (no motion module, F=1): native vs fp32 {rel(yn, y32):.2e}; fp16-eager vs fp32 {rel(y16, y32):.2e}")
    assert rel(yn, y32) <= rel(y16, y32) + 1e-4


def test_unet_full_width_against_reference_golden():
    g = torch.load(os.path.join(GOLD, "unet_full_tiny.pt"), weights_only=False)
    ora, nat = make_unet((320, 640, 1280, 1280), 768, seed=g["seed"])
    x, ehs, pose = g["x"].cuda().half(), g["ehs"].cuda().half(), g["pose"].cuda().half()
    with torch.no_grad():
        yn = nat(x, g["t"], ehs, pose_cond_fea=pose, return_dict=False)[0]
        y16 = ora.half()(x, torch.tensor(g["t"], device="cuda"), ehs, pose_cond_fea=pose)[0]
    gold = g["y"].cuda()  # fp32 output of the reference's own modules (fp32 weights, fp32 inputs)
    e_nat, e_ref = rel(yn, gold), rel(y16, gold)
    report(f"full-width tiny: native vs reference golden {e_nat:.2e}; fp16-eager vs golden {e_ref:.2e}")
    assert e_nat <= e_ref + 2e-4
    del ora, nat
    torch.cuda.empty_cache()


def make_writer(chs, xdim, seed=17):
    ora = O.synthetic_init(O.UNet2DConditionModel(block_out_channels=chs, cross_attention_dim=xdim).eval(), seed=seed).half().float().cuda()
    nat = hv.UNet2DConditionModel(block_out_channels=chs, cross_attention_dim=xdim)
    nat.load_state_dict(ora.state_dict())
    return ora, nat.to("cuda", torch.float16)


def reference_banks_fp32(g):
    """The writer's 16 banks in fp32 on the CPU: the golden file stores only a sample of them, and the oracle's fp32 CPU writer
    reproduces the reference's banks (tests/test_oracle_cpu.py pins it against that sample at 1e-5)."""
    w = O.synthetic_init(O.UNet2DConditionModel(block_out_channels=(64, 128, 256, 256), cross_attention_dim=64).eval(), seed=g["seed"])
    O.set_reference_write(w)
    with torch.no_grad():
        w(g["lat"], torch.tensor(0), g["ehs"])
    banks = O.written_banks(w)
    assert all(torch.allclose(b[:, r], gb, atol=1e-5, rtol=1e-5) for b, r, gb in zip(banks, g["bank_rows"], g["bank_samples"]))
    return banks


def test_reference_writer_unet2d_golden_banks_and_chain():
    """Native reference ("writer") UNet: hidden + 16 banks against vectors from the reference's own UNet2DConditionModel in write
    mode; then writer -> ReferenceAttentionControl.update -> native denoising UNet against the reference's chain."""
    g = torch.load(os.path.join(GOLD, "unet2d_writer_narrow.pt"), weights_only=False)
    ora, nat = make_writer((64, 128, 256, 256), 64, seed=g["seed"])
    lat, ehs = g["lat"].cuda().half(), g["ehs"].cuda().half()
    writer = hv.ReferenceAttentionControl(nat, do_classifier_free_guidance=True, mode="write", batch_size=1, fusion_blocks="full")
    with torch.no_grad():
        hid = nat(lat, torch.zeros((), dtype=torch.long, device="cuda"), encoder_hidden_states=ehs, return_dict=False)[0]
        hid16 = ora.half()(lat, torch.tensor(0, device="cuda"), ehs)[0]
        ora.float()
    banks = [b.bank[0] for b, _ in nat.writer_blocks()]
    assert hid.shape == (2, 64, 16, 16) and [tuple(b.shape) for b in banks] == [tuple(s) for s in g["bank_shapes"]]
    e_hid, e_ref = rel(hid, g["hidden"].cuda()), rel(hid16, g["hidden"].cuda())
    # the golden file keeps a fixed, seeded quarter of every bank's tokens
    e_banks = [rel(b[:, r.cuda()], gb.cuda()) for b, r, gb in zip(banks, g["bank_rows"], g["bank_samples"])]
    report(f"writer UNet2D: hidden native vs reference golden {e_hid:.2e} (fp16-eager {e_ref:.2e}); banks max {max(e_banks):.2e}")
    assert e_hid <= e_ref + 2e-4
    assert max(e_banks) <= 2e-3
    # writer -> reader on the native denoising UNet; reference chain value y3
    ora3, nat3 = make_unet((64, 128, 256, 256), 64, seed=g["seed3"])
    reader = hv.ReferenceAttentionControl(nat3, do_classifier_free_guidance=True, mode="read", batch_size=1, fusion_blocks="full")
    reader.update(writer)
    x3 = g["x3"].cuda().half()
    with torch.no_grad():
        y = nat3(x3, g["t3"], ehs, return_dict=False)[0]
        O.set_reference_banks(ora3, [gb.cuda().half() for gb in reference_banks_fp32(g)], cfg=True)
        y16 = ora3.half()(x3, torch.tensor(g["t3"], device="cuda"), ehs)[0]
    e_nat, e_16 = rel(y, g["y3"].cuda()), rel(y16, g["y3"].cuda())
    report(f"writer -> reader chain: native vs reference golden {e_nat:.2e} (fp16-eager {e_16:.2e})")
    assert e_nat <= e_16 + 2e-4
    reader.clear(); writer.clear()
    # without write mode the forward is unchanged and leaves no banks
    nat._ref_write = False
    with torch.no_grad():
        hid2 = nat(lat, 0, ehs, return_dict=False)[0]
    assert torch.equal(hid, hid2) and all(len(b.bank) == 0 for b, _ in nat.writer_blocks())


def test_reference_writer_unet2d_full_width_config2_shape():
    """SD1.5-width writer at the 96x72 latent of BASELINE config 2/3: bank shapes are what the reader takes, values vs the oracle."""
    ora, nat = make_writer((320, 640, 1280, 1280), 768, seed=17)
    g = torch.Generator(device="cuda").manual_seed(3)
    lat = torch.randn(1, 4, 96, 72, generator=g, device="cuda").half().repeat(2, 1, 1, 1)
    ehs = torch.cat([torch.zeros(1, 1, 768, device="cuda"), torch.randn(1, 1, 768, generator=g, device="cuda")]).half()
    hv.ReferenceAttentionControl(nat, do_classifier_free_guidance=True, mode="write", fusion_blocks="full")
    O.set_reference_write(ora)
    with torch.no_grad():
        hid = nat(lat, 0, ehs, return_dict=False)[0]
        hid32 = ora(lat.float(), torch.tensor(0, device="cuda"), ehs.float())[0]
    banks, banks32 = [b.bank[0] for b, _ in nat.writer_blocks()], O.written_banks(ora)
    assert [tuple(b.shape[1:]) for b in banks] == [(432, 1280)] * 5 + [(108, 1280)] + [(1728, 640)] * 5 + [(6912, 320)] * 5
    errs = [rel(a, b) for a, b in zip(banks, banks32)]
    report(f"writer UNet2D full width 96x72: hidden {rel(hid, hid32):.2e}, banks max {max(errs):.2e}")
    assert rel(hid, hid32) <= 2.5e-3 and max(errs) <= 2e-3
    assert torch.equal(banks[0][0], banks[0][0]) and torch.isfinite(hid).all()


def test_pose_guider_and_camera_encoder_golden():
    g = torch.load(os.path.join(GOLD, "pose_guider.pt"), weights_only=False)
    o = O.synthetic_init(O.PoseGuider().eval(), seed=g["seed"])
    pg = hv.PoseGuider(320, block_out_channels=(16, 32, 96, 256))
    pg.load_state_dict(o.state_dict())
    pg = pg.to("cuda", torch.float16)
    y = pg(g["x"].cuda().half())
    torch.cuda.synchronize()
    assert y.shape == g["y"].shape
    assert rel(y, g["y"].cuda()) < 1e-3
    g = torch.load(os.path.join(GOLD, "camera_encoder.pt"), weights_only=False)
    o = O.synthetic_init(O.CameraPoseEncoder().eval(), seed=g["seed"])
    cam = hv.CameraPoseEncoder(downscale_factor=8, channels=[320], nums_rb=2, cin=384, ksize=1, sk=True, use_conv=False, compression_factor=1,
                               temporal_attention_nhead=8, attention_block_types=["Temporal_Self"], temporal_position_encoding=True,
                               temporal_position_encoding_max_len=24)
    cam.load_state_dict(o.state_dict())
    cam = cam.to("cuda", torch.float16)
    y = cam(g["x"].cuda().half())[0]
    torch.cuda.synchronize()
    assert y.shape == g["y"].shape
    assert rel(y, g["y"].cuda()) < 1.5e-3


def test_camera_encoder_from_cameras_plucker_on_device():
    """SURVEY 8f-3: the Plucker embedding generated on the GPU inside the encoder's PixelUnshuffle producer, from the intrinsics / relative
    poses of a shipped camera trajectory (tests/golden/plucker.pt: rows of data/test_set/camera_test_set.zip and the reference's own
    Camera + ray_condition output), against (a) the golden embedding and (b) the encoder fed with that embedding."""
    import ctypes as C

    import torch.nn.functional as F

    from humanvid_b200 import _native as N
    from humanvid_b200 import camera as Cm

    g = torch.load(os.path.join(GOLD, "plucker.pt"), weights_only=False)
    img = tuple(g["img_size"])                               # (W, H) = (48, 64)
    cams = [Cm.Camera(r, "test", img) for r in g["rows"]]
    K, c2w = Cm.relative_cameras(cams, 0, list(range(1, 9)), img)
    Fr, H, W = 8, img[1], img[0]
    gold = g["y"].cuda()                                     # (1, 8, 6, 64, 48) fp16, the reference's ray_condition output
    un = torch.zeros(Fr, H // 8, W // 8, 384, device="cuda", dtype=torch.half)
    Kd, Md = K.cuda().contiguous(), c2w.cuda().contiguous()   # (kept referenced: the launch is asynchronous)
    N.check(N.lib().hv_op_plucker_unshuffle(N.ptr(Kd), N.ptr(Md), N.ptr(un), N.i64(Fr), N.i64(H), N.i64(W), N.i32(8), N.stream()))
    ref_un = F.pixel_unshuffle(gold[0], 8).permute(0, 2, 3, 1).contiguous()
    torch.cuda.synchronize()
    e_embed = rel(un, ref_un)
    o = O.synthetic_init(O.CameraPoseEncoder().eval(), seed=13)
    cam = hv.CameraPoseEncoder(downscale_factor=8, channels=[320], nums_rb=2, cin=384, ksize=1, sk=True, use_conv=False, compression_factor=1,
                               temporal_attention_nhead=8, attention_block_types=["Temporal_Self"], temporal_position_encoding=True,
                               temporal_position_encoding_max_len=24)
    cam.load_state_dict(o.state_dict())
    cam = cam.to("cuda", torch.float16)
    y_img = cam(gold.transpose(1, 2).contiguous())[0]        # (1, 6, 8, H, W) like scripts/pose2vid.py:285 hands it to the pipeline
    y_cam = cam.forward_cameras(K, c2w, H, W)[0]
    torch.cuda.synchronize()
    report(f"plucker on device: embedding vs reference golden {e_embed:.2e}; encoder output vs embedding-fed encoder {rel(y_cam, y_img):.2e}")
    assert (un.float() - ref_un.float()).abs().max() <= 2e-3 and e_embed < 3e-4      # fp32 ray arithmetic, differences of one fp16 ulp
    assert y_cam.shape == y_img.shape and rel(y_cam, y_img) < 1e-3


def test_pose_guider_config2_shape_vs_oracle_fp16():
    o = O.synthetic_init(O.PoseGuider().eval(), seed=3).half().cuda()
    pg = hv.PoseGuider(320, block_out_channels=(16, 32, 96, 256))
    pg.load_state_dict(o.state_dict())
    pg = pg.to("cuda", torch.float16)
    x = torch.rand(1, 3, 4, 768, 576, device="cuda").half()
    with torch.no_grad():
        ref = o.float()(x.float())
        y = pg(x)
    torch.cuda.synchronize()
    assert y.shape == (1, 320, 4, 96, 72)
    assert rel(y, ref) < 1e-3


def test_zero_init_modules_are_exact_noops():
    # reference zero-inits kept (pose_guider.py:42, pose_adaptor.py:217): outputs must be exactly zero
    pg = hv.PoseGuider(320, block_out_channels=(16, 32, 96, 256)).to("cuda", torch.float16)
    y = pg(torch.rand(1, 3, 2, 64, 64, device="cuda").half())
    assert float(y.abs().max()) == 0.0
    cam = hv.CameraPoseEncoder(downscale_factor=8, channels=[320], nums_rb=2, cin=384, ksize=1, sk=True, use_conv=False, compression_factor=1,
                               temporal_attention_nhead=8, attention_block_types=["Temporal_Self"], temporal_position_encoding=True,
                               temporal_position_encoding_max_len=24).to("cuda", torch.float16)
    y = cam(torch.randn(1, 6, 2, 64, 64, device="cuda").half())[0]
    assert float(y.abs().max()) == 0.0


def test_too_many_frames_is_an_error(narrow):
    _, nat = narrow
    x, ehs, pose = unet_inputs(2, 33, 16, 16, 64, 64)
    with pytest.raises(RuntimeError, match="max_len"):
        nat(x, 10, ehs, pose_cond_fea=pose)


def test_registered_reader_with_empty_banks_warns_once():
    # VERDICT r1 item 9: a reader control without a written bank must not be silent
    _, nat = make_unet((64, 128, 256, 256), 64, seed=5)
    hv.ReferenceAttentionControl(nat, mode="read", do_classifier_free_guidance=True, fusion_blocks="full")
    x, ehs, pose = unet_inputs(2, 4, 16, 16, 64, 64)
    with pytest.warns(RuntimeWarning, match="reference bank is empty"):
        nat(x, 10, ehs, pose_cond_fea=pose)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        nat(x, 11, ehs, pose_cond_fea=pose)   # once per model
