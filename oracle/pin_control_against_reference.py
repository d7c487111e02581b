"""Record how the reference's OWN ReferenceAttentionControl (src/models/mutual_self_attention.py) drives the native UNets, for
tests/test_reference_control_cpu.py.

Run with a checkout of the reference tree (pin_against_reference.REF):

    python oracle/pin_control_against_reference.py        # (re)write tests/golden/reference_control.json

The reference's control finds its blocks with isinstance() against src/models/attention.py's classes (mutual_self_attention.py:284-300,
321-330); the native blocks adopt those classes when they are loaded.  Every writer block of a native UNet2DConditionModel is given a
bank holding its own index, the reference's reader runs update(writer) on a native UNet3DConditionModel, and what each reader block
received is written down by module name: the pairing of reader and writer blocks, the dtype of the handed-over bank, and the order in
which the reference's reader ranks its blocks (its attn_weight = i / n).
"""
from __future__ import annotations

import json
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import pin_against_reference as P  # noqa: E402  (the stand-ins for the diffusers symbols the reference imports)

GOLD = os.path.join(ROOT, "tests", "golden")
MM = dict(num_attention_heads=8, num_transformer_block=1, attention_block_types=["Temporal_Self", "Temporal_Self"], temporal_position_encoding=True,
          temporal_position_encoding_max_len=32, temporal_attention_dim_div=1)


def build_unets(hv):
    """The UNet pair of tests/test_reference_control_cpu.py."""
    unet = hv.UNet3DConditionModel(block_out_channels=(32, 64, 64, 64), cross_attention_dim=32, use_motion_module=True, use_inflated_groupnorm=True,
                                   motion_module_resolutions=(1, 2, 4, 8), motion_module_mid_block=True, motion_module_type="Vanilla", motion_module_kwargs=MM)
    wr = hv.UNet2DConditionModel(block_out_channels=(32, 64, 64, 64), cross_attention_dim=32)
    return unet, wr


def main():
    P.install_stubs()
    P.install_stubs_2d()
    from src.models.mutual_self_attention import ReferenceAttentionControl as RefControl   # the reference's class, unmodified

    import humanvid_b200 as hv

    unet, wr = build_unets(hv)
    writer = RefControl(wr, do_classifier_free_guidance=True, mode="write", batch_size=1, fusion_blocks="full")
    reader = RefControl(unet, do_classifier_free_guidance=True, mode="read", batch_size=1, fusion_blocks="full")
    writers = [(n, m) for n, m in wr.named_modules() if hasattr(m, "bank")]
    for i, (_, m) in enumerate(writers):
        m.bank.append(torch.full((2, 3, m.norm1.normalized_shape[0]), float(i)))
    reader.update(writer)
    readers = [(n, m) for n, m in unet.named_modules() if hasattr(m, "bank")]
    out = {"reader_order": [n for n, m in sorted(readers, key=lambda nm: nm[1].attn_weight)],
           "pairing": {n: writers[int(m.bank[0][0, 0, 0])][0] for n, m in readers},
           "bank_dtype": str(readers[0][1].bank[0].dtype)}
    assert len(readers) == len(writers) == 16 and all(len(m.bank) == 1 and str(m.bank[0].dtype) == out["bank_dtype"] for _, m in readers)
    reader.clear()
    writer.clear()
    assert all(len(m.bank) == 0 for _, m in readers)
    with open(os.path.join(GOLD, "reference_control.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
