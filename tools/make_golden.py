#!/usr/bin/env python
"""Generate tests/golden/*.pt by EXECUTING the reference's own torch-only modules (build container only).

The reference (jianzongwu/DiffSensei @ /root/reference) has no tests or golden vectors (SURVEY.md §4).
Two of its hot-path files import nothing but torch, so they run here on CPU:
    src/models/attention_processor.py   (AttnProcessor2_0, MaskedIPAttnProcessor2_0)
    src/models/resampler.py             (Resampler)
and ``UNetMangaModel.encode_dialog_bbox`` (src/models/unet.py:88-114) is a pure-torch method that is lifted
out of its (diffusers-dependent) module with ``ast`` and executed on a stub ``self``.
Nothing is copied into this repository: the reference code is imported/executed from where it lies and only
its seeded inputs and outputs are saved.  /root/reference does not exist on the GPU box, so the fixtures are
committed; re-run this script only in the build container:

    python tools/make_golden.py
"""
from __future__ import annotations

import ast
import importlib.util
import os
import sys
import types

import torch

REF = "/root/reference"
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def load_module(name: str, path: str):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def lift_function(path: str, func_name: str):
    """Compile one function definition out of a module that cannot be imported (missing diffusers)."""
    tree = ast.parse(open(path).read())
    for node in ast.walk(tree):
        if isinstance(node, ast.FunctionDef) and node.name == func_name:
            mod = ast.Module(body=[node], type_ignores=[])
            ns = {"torch": torch}
            exec(compile(mod, path, "exec"), ns)
            return ns[func_name]
    raise KeyError(func_name)


class StubAttn:
    """The attributes a processor reads from diffusers' Attention (attention_processor.py:34-94) for SDXL."""

    def __init__(self, dim, kv_dim, heads, gen):
        def lin(i, o, bias):
            m = torch.nn.Linear(i, o, bias=bias)
            with torch.no_grad():
                m.weight.copy_(torch.randn(o, i, generator=gen) / i ** 0.5)
                if bias:
                    m.bias.copy_(torch.randn(o, generator=gen) * 0.1)
            return m

        self.heads = heads
        self.spatial_norm = None
        self.group_norm = None
        self.norm_cross = False
        self.residual_connection = False
        self.rescale_output_factor = 1.0
        self.to_q = lin(dim, dim, False)
        self.to_k = lin(kv_dim, dim, False)
        self.to_v = lin(kv_dim, dim, False)
        self.to_out = [lin(dim, dim, True), torch.nn.Identity()]

    def weights(self):
        return {"to_q": self.to_q.weight.detach().clone(), "to_k": self.to_k.weight.detach().clone(),
                "to_v": self.to_v.weight.detach().clone(), "to_out_w": self.to_out[0].weight.detach().clone(),
                "to_out_b": self.to_out[0].bias.detach().clone()}


SAMPLE = 4096


def sampled(case, **outputs):
    """``case`` plus the outputs: whole when small, else the elements at one fixed, seeded sample of SAMPLE flat
    indices (``case["idx"]``, shared by all outputs of the case) so that every fixture stays well under 1 MB."""
    numel = next(iter(outputs.values())).numel()
    if numel > SAMPLE:
        idx = torch.randperm(numel, generator=torch.Generator().manual_seed(7))[:SAMPLE].sort().values.to(torch.int32)
        case["idx"] = idx
        outputs = {k: v.flatten()[idx.long()].clone() for k, v in outputs.items()}
    return {**case, **outputs}


@torch.no_grad()
def main():
    os.makedirs(OUT, exist_ok=True)
    ap = load_module("ref_attention_processor", f"{REF}/src/models/attention_processor.py")
    rs = load_module("ref_resampler", f"{REF}/src/models/resampler.py")

    # ------------------------------------------------------------------ self-attention
    g = torch.Generator().manual_seed(0)
    attn = StubAttn(128, 128, 2, g)
    hs = torch.randn(2, 96, 128, generator=g)
    out = ap.AttnProcessor2_0()(attn, hs)
    torch.save({"hs": hs, "heads": 2, **attn.weights(), "out": out}, f"{OUT}/attn_self.pt")

    # ------------------------------------------------------------------ text + masked-IP cross-attention
    g = torch.Generator().manual_seed(1)
    dim, kv, heads, n_ips, tpi = 128, 64, 2, 4, 16
    H, W = 12, 20                               # feature map; aspect_ratio = H / W as pipeline :272
    attn = StubAttn(dim, kv, heads, g)
    proc = ap.MaskedIPAttnProcessor2_0(hidden_size=dim, cross_attention_dim=kv, num_ip_tokens=n_ips * tpi,
                                       num_dummy_tokens=tpi)
    proc.to_k_ip.weight.copy_(torch.randn(dim, kv, generator=g) / kv ** 0.5)
    proc.to_v_ip.weight.copy_(torch.randn(dim, kv, generator=g) / kv ** 0.5)
    proc.scale = 0.6
    hs = torch.randn(2, H * W, dim, generator=g)
    ehs = torch.randn(2, 77 + 80, kv, generator=g)
    bbox = torch.tensor([[[0.0, 0.0, 0.0, 0.0]] * 4,
                         [[0.05, 0.10, 0.50, 0.95], [0.50, 0.15, 0.95, 0.90], [0.30, 0.55, 0.70, 1.0],
                          [0.0, 0.0, 0.0, 0.0]]])
    out = proc(attn, hs, encoder_hidden_states=ehs, bbox=bbox, aspect_ratio=H / W)
    torch.save({"hs": hs, "ehs": ehs, "bbox": bbox, "aspect_ratio": H / W, "heads": heads, "scale": 0.6,
                "num_ip_tokens": n_ips * tpi, "num_dummy": tpi, **attn.weights(),
                "to_k_ip": proc.to_k_ip.weight.detach().clone(), "to_v_ip": proc.to_v_ip.weight.detach().clone(),
                "out": out}, f"{OUT}/attn_cross_ip.pt")

    # ------------------------------------------------------------------ IP mask known-answer tests
    proc = ap.MaskedIPAttnProcessor2_0(hidden_size=64, cross_attention_dim=64, num_ip_tokens=64, num_dummy_tokens=16)
    kats = []
    # (iii) of SURVEY.md §8c: open fraction 0.2065 at N = 32x32
    bb = torch.tensor([[[0.0] * 4] * 4, [[.1, .1, .6, .9], [.5, .2, 1, 1], [0.0] * 4, [0.0] * 4]])
    for (n, ar, b) in [(1024, 1.0, bb), (24 * 11, 184 / 352, bb), (15 * 5, 136 / 480, bb), (38 * 27, 27 / 38, bb),
                       (64, 1.0, torch.tensor([[[0.5, 0.5, 0.5, 0.5], [0.0, 0.0, 1.0, 1.0], [3 / 7, 0.0, 4 / 7, 1.0],
                                               [0.25, 0.25, 0.75, 0.75]]]))]:
        m = proc.prepare_attention_mask_ip(b, torch.zeros(b.shape[0], n, 64), 1, ar)[:, 0]   # heads identical
        kats.append({"N": n, "aspect_ratio": ar, "bbox": b, "open": (m == 0)})
    torch.save(kats, f"{OUT}/ip_mask_kats.pt")

    # derived (H', W') for every (bucket, level): with bbox [0,0,1,0] only the first row (y == 0) is inside,
    # so the number of open ip-0 keys' pixels equals the derived width.
    try:
        du = load_module("ref_dataset_utils", f"{REF}/src/datasets/utils.py")
        buckets = [b for grp in du.size_buckets for b in grp["buckets"]]
    except Exception as e:  # PIL missing etc.: parse the literal instead
        src = open(f"{REF}/src/datasets/utils.py").read()
        tree = ast.parse(src)
        lit = next(n.value for n in tree.body if isinstance(n, ast.Assign) and n.targets[0].id == "size_buckets")
        buckets = [b for grp in ast.literal_eval(lit) for b in grp["buckets"]]
    rows = []
    row_box = torch.tensor([[[0.0, 0.0, 1.0, 0.0]] + [[0.0] * 4] * 3])
    for (bh, bw, _r) in buckets:
        for down in (16, 32):                       # level-1 and level-2 feature maps (latent/2, latent/4)
            lh, lw = bh // 8, bw // 8               # latent size
            # true feature-map dims after stride-2 convs with padding 1: ceil division
            fh, fw = lh, lw
            for _ in range({16: 1, 32: 2}[down]):
                fh, fw = (fh - 1) // 2 + 1, (fw - 1) // 2 + 1
            n = fh * fw
            ar = lh / lw                            # pipeline_diffsensei.py:272 uses the LATENT aspect ratio
            m = proc.prepare_attention_mask_ip(row_box, torch.zeros(1, n, 64), 1, ar)[0, 0]
            w_derived = int((m[:, 16] == 0).sum())
            rows.append((bh, bw, down, fh, fw, n // w_derived, w_derived))
    torch.save(torch.tensor(rows, dtype=torch.int32), f"{OUT}/derived_hw_table.pt")
    mism = sum(1 for r in rows if (r[3], r[4]) != (r[5], r[6]))
    print(f"derived-(H',W') table: {len(rows)} (bucket, level) rows, {mism} differ from the true feature map")

    # ------------------------------------------------------------------ dialog bbox embedding
    enc = lift_function(f"{REF}/src/models/unet.py", "encode_dialog_bbox")
    g = torch.Generator().manual_seed(2)
    cases = []
    for dtype in (torch.float32, torch.bfloat16):
        stub = types.SimpleNamespace(dialog_bbox_embedding=torch.randn(8, generator=g).to(dtype))
        sample = torch.randn(2, 8, 19, 152, generator=g).to(dtype)
        db = torch.tensor([[[.05, .05, .30, .20], [.70, .05, .95, .22], [.40, .80, .65, .97], [0.0, 0.0, 0.9, 0.5]]
                           + [[0.0] * 4] * 4, [[0.0] * 4] * 8]).to(dtype)
        cases.append({"sample": sample, "dialog_bbox": db, "emb": stub.dialog_bbox_embedding,
                      "out": enc(stub, sample, db)})
    torch.save(cases, f"{OUT}/dialog_embed.pt")

    # ------------------------------------------------------------------ Resampler (tiny and SHIPPED config)
    # shipped = configs/model/diffsensei.yaml + scripts/demo/gradio_wo_mllm.py:174-185: 83,978,752 params.  The weights
    # and inputs are NOT stored: both sides regenerate them from the seeds below with
    # diffsensei_b200.weights.random_state_dict / torch.Generator (tests/test_oracle_golden.py::resampler_case); only
    # the reference's outputs are committed, a seeded sample of them where they are large.
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from diffsensei_b200.config import RESAMPLER, RESAMPLER_TINY
    from diffsensei_b200.weights import random_state_dict, resampler_param_shapes
    import dataclasses
    for fname, rc, wseed, iseed, n_tokens, n_real in (("resampler_tiny.pt", RESAMPLER_TINY, 3, 4, 33, 2),
                                                      ("resampler_full.pt", RESAMPLER, 42, 43, 257, 3)):
        kwr = dataclasses.asdict(rc)
        model = rs.Resampler(**kwr).eval()
        print(f"Resampler({fname}) params:", sum(p.numel() for p in model.parameters()))
        sdr = random_state_dict(resampler_param_shapes(rc), seed=wseed, device="cpu")
        sdr = {k: v.to(torch.bfloat16).float() for k, v in sdr.items()}      # bf16-representable on both sides
        model.load_state_dict(sdr)
        gx = torch.Generator().manual_seed(iseed)
        x = torch.randn(1, 4, n_tokens, rc.embedding_dim, generator=gx).to(torch.bfloat16).float()
        magi = torch.randn(1, 4, rc.magi_embedding_dim, generator=gx).to(torch.bfloat16).float()
        x[0, n_real:] = 0                                                    # real characters, the rest padded (:131-132)
        magi[0, n_real:] = 0
        case = {"kwargs": kwr, "weight_seed": wseed, "input_seed": iseed, "n_tokens": n_tokens, "n_real": n_real}
        torch.save(sampled(case, out=model(x, magi), out_zero=model(torch.zeros_like(x), torch.zeros_like(magi))),
                   f"{OUT}/{fname}")
    # ------------------------------------------------------------------ QwenResampler (MLLM adaptor, §8f-4)
    # configs/model/diffsensei.yaml agent.input_resampler / output_resampler + a small one; weights / inputs are
    # regenerated from seeds on both sides (tests/test_oracle_golden.py::qwen_case), only outputs are stored
    qr = load_module("ref_qwen_resampler", f"{REF}/src/models/qwen_resampler.py")
    qcases = {}
    for name, kw in (("tiny", dict(grid_size=4, embed_dim=128, num_heads=2, kv_dim=64)),
                     ("input", dict(grid_size=8, embed_dim=5120, num_heads=32, kv_dim=2048)),
                     ("output", dict(grid_size=8, embed_dim=2048, num_heads=32, kv_dim=5120))):
        m = qr.QwenResampler(**kw).eval()
        gq = torch.Generator().manual_seed(50)
        sdq = {}
        for k, v in m.state_dict().items():
            if k == "pos_embed":
                sdq[k] = v
            elif k.endswith("weight") and v.dim() == 1:
                sdq[k] = (1 + 0.1 * torch.randn(v.shape, generator=gq)).to(torch.bfloat16).float()
            elif k.endswith("bias"):
                sdq[k] = (0.05 * torch.randn(v.shape, generator=gq)).to(torch.bfloat16).float()
            elif k == "query":
                sdq[k] = torch.randn(v.shape, generator=gq).to(torch.bfloat16).float()
            else:
                sdq[k] = (torch.randn(v.shape, generator=gq) * v.shape[-1] ** -0.5).to(torch.bfloat16).float()
        m.load_state_dict(sdq)
        xq = torch.randn(2, kw["grid_size"] ** 2, kw["kv_dim"], generator=gq).to(torch.bfloat16).float()
        qcases[name] = sampled({"kwargs": kw, "seed": 50}, out=m(xq))
    torch.save(qcases, f"{OUT}/qwen_resampler.pt")
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    sys.exit(main())
