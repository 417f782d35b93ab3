"""Pin the oracle restatement to the EXECUTED reference (tests/golden/*.pt, made by tools/make_golden.py from
/root/reference's own attention_processor.py / resampler.py / encode_dialog_bbox).  CPU only."""
import os

import pytest
import torch

from conftest import GOLDEN, rel_l2
from oracle import attention as A
from oracle.resampler import OracleResampler
from oracle.unet import dialog_boxes_to_pixels, encode_dialog_bbox


def _load(name):
    return torch.load(os.path.join(GOLDEN, name), weights_only=False)


def test_self_attention_matches_reference():
    g = _load("attn_self.pt")
    out = A.self_attention(g["hs"], g["to_q"], g["to_k"], g["to_v"], g["to_out_w"], g["to_out_b"], g["heads"])
    assert rel_l2(out, g["out"]) < 1e-5


def test_cross_ip_attention_matches_reference():
    g = _load("attn_cross_ip.pt")
    out = A.cross_ip_attention(g["hs"], g["ehs"], g["bbox"], g["aspect_ratio"], g["to_q"], g["to_k"], g["to_v"],
                               g["to_k_ip"], g["to_v_ip"], g["to_out_w"], g["to_out_b"], g["heads"], g["scale"],
                               g["num_ip_tokens"], g["num_dummy"])
    assert rel_l2(out, g["out"]) < 1e-5


def test_blend_happens_before_out_projection():
    # SURVEY §8c KAT (vi): hs + scale*ip_hs BEFORE to_out  => output is affine in `scale` with the bias counted once
    g = _load("attn_cross_ip.pt")
    f = lambda s: A.cross_ip_attention(g["hs"], g["ehs"], g["bbox"], g["aspect_ratio"], g["to_q"], g["to_k"],
                                       g["to_v"], g["to_k_ip"], g["to_v_ip"], g["to_out_w"], g["to_out_b"],
                                       g["heads"], s, g["num_ip_tokens"], g["num_dummy"])
    o0, o1, o2 = f(0.0), f(1.0), f(2.0)
    assert rel_l2(o2 - o1, o1 - o0) < 1e-4


def test_ip_mask_kats_bit_exact():
    for kat in _load("ip_mask_kats.pt"):
        bb = kat["bbox"]
        open_ = A.ip_open_mask(bb, kat["N"], kat["aspect_ratio"], 16, 16)
        assert torch.equal(open_, kat["open"]), (kat["N"], kat["aspect_ratio"])


def test_ip_mask_probed_invariants():
    kats = _load("ip_mask_kats.pt")
    k = kats[0]                                   # N = 32x32, SURVEY §8c (iii)
    assert abs(k["open"].float().mean().item() - 0.2065) < 5e-4
    neg = k["open"][0]                            # all-zero boxes: pixel 0 sees the 64 ip keys, not the dummies
    assert neg[0, 16:].all() and not neg[0, :16].any()
    assert neg[1:, :16].all() and not neg[1:, 16:].any()
    assert (k["open"].sum(-1) >= 16).all()        # every query keeps >= 16 open keys


def test_derived_hw_table():
    tab = _load("derived_hw_table.pt")
    assert tab.shape == (198, 7)
    mism = 0
    for bh, bw, _down, fh, fw, dh, dw in tab.tolist():
        h, w = A.derive_hw(fh * fw, (bh // 8) / (bw // 8))
        assert (h, w) == (dh, dw)
        mism += (fh, fw) != (dh, dw)
    assert mism == 5                              # SURVEY §3.4: 5/198 (bucket, level) cases differ
    rows = {(r[0], r[1], r[2]): (r[5], r[6]) for r in tab.tolist()}
    assert rows[(352, 184, 16)] == (24, 11) and rows[(136, 480, 32)] == (3, 25)


def test_dialog_embed_matches_reference_including_bf16_truncation():
    for case in _load("dialog_embed.pt"):
        out = encode_dialog_bbox(case["sample"], case["dialog_bbox"], case["emb"])
        assert torch.equal(out, case["out"])
    bf = torch.tensor([0.0, 0.0, 0.9, 0.5], dtype=torch.bfloat16)
    assert dialog_boxes_to_pixels(bf.unsqueeze(0), 19, 152)[0][2] == 137     # int(bf16(0.9)*152) = 137
    assert dialog_boxes_to_pixels(bf.float().unsqueeze(0) * 0 + torch.tensor([0, 0, 0.9, 0.5]), 19, 152)[0][2] == 136


def sampled(t, g):
    """The elements of ``t`` a fixture stores: the seeded sample ``g["idx"]`` of a large output, else ``t`` whole."""
    return t.flatten()[g["idx"].long()] if "idx" in g else t


def resampler_case(name):
    """Regenerate the weights / inputs of tests/golden/<name> from its seeds (tools/make_golden.py)."""
    from diffsensei_b200.config import ResamplerConfig
    from diffsensei_b200.weights import random_state_dict, resampler_param_shapes
    g = _load(name)
    rc = ResamplerConfig(**g["kwargs"])
    sd = random_state_dict(resampler_param_shapes(rc), seed=g["weight_seed"], device="cpu")
    sd = {k: v.to(torch.bfloat16).float() for k, v in sd.items()}
    gx = torch.Generator().manual_seed(g["input_seed"])
    x = torch.randn(1, 4, g["n_tokens"], rc.embedding_dim, generator=gx).to(torch.bfloat16).float()
    magi = torch.randn(1, 4, rc.magi_embedding_dim, generator=gx).to(torch.bfloat16).float()
    x[0, g["n_real"]:] = 0
    magi[0, g["n_real"]:] = 0
    return g, sd, x, magi


def test_resampler_matches_reference():
    g, sd, x, magi = resampler_case("resampler_tiny.pt")
    m = OracleResampler(**g["kwargs"]).eval()
    m.load_state_dict(sd)
    with torch.no_grad():
        out = m(x, magi)
        assert rel_l2(sampled(out, g), g["out"]) < 1e-5
        assert rel_l2(sampled(m(torch.zeros_like(x), torch.zeros_like(magi)), g), g["out_zero"]) < 1e-5
    assert out.shape == (1, 80, 128)


def test_resampler_shipped_config_param_count():
    from diffsensei_b200.config import RESAMPLER
    from diffsensei_b200.weights import resampler_param_shapes
    n = sum(torch.Size(s).numel() for s in resampler_param_shapes(RESAMPLER).values())
    assert n == 83_978_752                        # SURVEY §8c (v)


def test_resampler_shipped_config_matches_executed_reference():
    """configs/model/diffsensei.yaml Resampler (dim 1280, depth 4, 20 heads, 257 CLIP tokens + 1 Magi token per
    character, 83,978,752 params): oracle restatement vs the reference's own resampler.py executed on the same
    seeded weights / inputs."""
    import dataclasses
    from diffsensei_b200.config import RESAMPLER
    g, sd, x, magi = resampler_case("resampler_full.pt")
    assert g["kwargs"] == dataclasses.asdict(RESAMPLER)
    m = OracleResampler(**g["kwargs"]).eval()
    m.load_state_dict(sd)
    assert sum(p.numel() for p in m.parameters()) == 83_978_752
    with torch.no_grad():
        assert rel_l2(sampled(m(x, magi), g), g["out"]) < 1e-5
        assert rel_l2(sampled(m(torch.zeros_like(x), torch.zeros_like(magi)), g), g["out_zero"]) < 1e-5


@pytest.mark.parametrize("name", ["tiny", "input", "output"])
def test_qwen_resampler_oracle_matches_executed_reference(name):
    """MLLM adaptor resampler (src/models/qwen_resampler.py:87-145) at a tiny config and at the two shipped ones
    (configs/model/diffsensei.yaml agent.input_resampler / output_resampler): restatement vs the executed reference."""
    from oracle.qwen_resampler import seeded_case
    g = _load("qwen_resampler.pt")[name]
    m, _sd, x = seeded_case(g["kwargs"], g["seed"])
    assert rel_l2(sampled(m(x), g), g["out"]) < 1e-5
