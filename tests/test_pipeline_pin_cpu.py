"""humanvid_b200/pipeline.py's host loop against the reference's OWN pipeline files (oracle/pin_pipeline_against_reference.py): both
pipelines drive the same module objects on CPU, so every difference would be the pipeline's.  The committed report of that run
(tests/golden/pipeline_pin_report.json) is checked, and the pipeline is run again against the reference pipeline's stored outputs."""
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REPORT = os.path.join(ROOT, "tests", "golden", "pipeline_pin_report.json")
EXACT = ["video_cfg_two_windows", "video_no_cfg_two_windows_sum_quirk", "video_cfg_single_window", "video_cfg_three_steps",
         "video_cfg_interpolation_factor_2_slerp", "video_cfg_interpolation_factor_3_linear", "video_cfg_with_callback", "callback_latents",
         "image_cfg", "image_no_cfg"]


def test_committed_pipeline_pin_report_is_exact():
    rep = json.load(open(REPORT))
    for k in EXACT:
        assert rep[k] == 0.0, (k, rep[k])
    assert rep["video_cfg_decode_batch_8"] <= 1e-6
    assert rep["decode_calls_reference_then_native"] == [[1] * 12, [8, 4]]      # the reference decodes frame by frame, SURVEY 8f-4 batches by 8
    assert rep["windows_12_8_2"] == [list(range(8)), [6, 7, 8, 9, 10, 11, 0, 1]]
    # the documented deviation: the reference's callback index is clobbered by its window-batching loop (pipeline_pose2vid_long.py:511-517)
    assert rep["callback_step_index_reference"] == [1, 1] and rep["callback_step_index_native"] == [0, 1] and rep["callback_timesteps_equal"]


def test_pipeline_matches_the_reference_pipeline():
    """Every case of the pinning run with this package's pipeline on the oracle's modules, against the stored outputs of the
    reference's own pipeline (tests/golden/pipeline_reference_outputs.pt)."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")   # the pipeline runs on the GPU when it sees one; the stored outputs are of a CPU fp32 run
    r = subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "pin_pipeline_against_reference.py"), "--against-golden"], capture_output=True,
                       text=True, timeout=900, cwd=ROOT, env=env)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "against golden OK" in r.stdout


def test_scheduler_step_signature_of_diffusers():
    """pipeline_pose2img.py:351-353 calls ``scheduler.step(..., eta=..., generator=..., return_dict=False)[0]``."""
    from humanvid_b200.scheduler import DDIMScheduler

    s = DDIMScheduler()
    s.set_timesteps(25)
    x, v = torch.randn(1, 4, 1, 8, 8), torch.randn(1, 4, 1, 8, 8)
    a = s.step(v, int(s.timesteps[0]), x, eta=0.0, generator=None).prev_sample
    b = s.step(v, s.timesteps[0], x, eta=0.0, generator=None, return_dict=False)
    assert isinstance(b, tuple) and torch.equal(a, b[0])
    with pytest.raises(NotImplementedError):
        s.step(v, 999, x, eta=0.5)
