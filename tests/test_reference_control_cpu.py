"""The reference's own ReferenceAttentionControl finds its blocks with isinstance() against src/models/attention.py's classes
(mutual_self_attention.py:284-300, 321-330).  A native UNet built inside the reference tree must therefore present blocks that
pass that test, or reader.update(writer) would silently zip nothing.  The tests run in a subprocess because the first plants a
module named ``src.models.attention`` in sys.modules."""
import os
import subprocess
import sys
import textwrap

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

COMMON = """
import sys, types
sys.path.insert(0, %r)
import torch, torch.nn as nn
MM = dict(num_attention_heads=8, num_transformer_block=1, attention_block_types=["Temporal_Self", "Temporal_Self"], temporal_position_encoding=True,
          temporal_position_encoding_max_len=32, temporal_attention_dim_div=1)
def build(hv):
    unet = hv.UNet3DConditionModel(block_out_channels=(32, 64, 64, 64), cross_attention_dim=32, use_motion_module=True, use_inflated_groupnorm=True,
                                   motion_module_resolutions=(1, 2, 4, 8), motion_module_mid_block=True, motion_module_type="Vanilla", motion_module_kwargs=MM)
    wr = hv.UNet2DConditionModel(block_out_channels=(32, 64, 64, 64), cross_attention_dim=32)
    return unet, wr
""" % ROOT


def _run(body):
    r = subprocess.run([sys.executable, "-c", COMMON + textwrap.dedent(body)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    return r.stdout


def test_blocks_adopt_a_loaded_reference_class():
    out = _run("""
        fake = types.ModuleType("src.models.attention")
        class TemporalBasicTransformerBlock(nn.Module):
            def __init__(self, dim, heads, head_dim):      # a constructor the shells could never call
                super().__init__()
        class BasicTransformerBlock(nn.Module):
            def __init__(self, dim, heads, head_dim):
                super().__init__()
        fake.TemporalBasicTransformerBlock, fake.BasicTransformerBlock = TemporalBasicTransformerBlock, BasicTransformerBlock
        for n in ("src", "src.models"):
            sys.modules.setdefault(n, types.ModuleType(n))
        sys.modules["src.models.attention"] = fake
        import humanvid_b200 as hv
        unet, wr = build(hv)
        def dfs(m):
            out = [m]
            for c in m.children():
                out += dfs(c)
            return out
        readers = [m for m in dfs(unet) if isinstance(m, fake.TemporalBasicTransformerBlock)]
        writers = [m for m in dfs(wr) if isinstance(m, fake.BasicTransformerBlock)]
        assert len(readers) == 16 and len(writers) == 16, (len(readers), len(writers))
        assert sorted(readers, key=lambda m: -m.norm1.normalized_shape[0]) == unet.reader_blocks()
        assert all(isinstance(m, hv.TemporalBasicTransformerBlock) for m in readers)
        assert set(unet.state_dict()) == set(build(hv)[0].state_dict())
        print("adopted", len(readers))
    """)
    assert "adopted 16" in out


def test_the_references_own_control_drives_the_native_unets():
    """tests/golden/reference_control.json is what the reference's own ReferenceAttentionControl did to these two UNets
    (oracle/pin_control_against_reference.py): the order it ranks the reader blocks in, which writer bank each reader block receives,
    and the bank dtype.  The native control must hand over the same banks the same way."""
    out = _run("""
        import json
        import humanvid_b200 as hv
        gold = json.load(open(%r))
        unet, wr = build(hv)
        writer = hv.ReferenceAttentionControl(wr, do_classifier_free_guidance=True, mode="write", batch_size=1, fusion_blocks="full")
        reader = hv.ReferenceAttentionControl(unet, do_classifier_free_guidance=True, mode="read", batch_size=1, fusion_blocks="full")
        # every writer block leaves a bank holding its own index
        writers = [(n, m) for n, m in wr.named_modules() if hasattr(m, "bank")]
        for i, (_, m) in enumerate(writers):
            m.bank.append(torch.full((2, 3, m.norm1.normalized_shape[0]), float(i)))
        reader.update(writer)
        readers = [(n, m) for n, m in unet.named_modules() if hasattr(m, "bank")]
        names = {id(m): n for n, m in readers}
        assert len(readers) == len(writers) == 16
        assert [names[id(m)] for m in unet.reader_blocks()] == gold["reader_order"]
        assert {n: writers[int(m.bank[0][0, 0, 0])][0] for n, m in readers} == gold["pairing"]
        assert all(len(m.bank) == 1 and str(m.bank[0].dtype) == gold["bank_dtype"] for _, m in readers)
        reader.clear()
        writer.clear()
        assert all(len(m.bank) == 0 for _, m in readers)
        print("reference control ok")
    """ % os.path.join(ROOT, "tests", "golden", "reference_control.json"))
    assert "reference control ok" in out
