"""TEST INFRASTRUCTURE ONLY.  Golden vectors for videoswap_b200/formats.py (SURVEY.md 8f-4, data formats), produced by the
REFERENCE's own functions read from /root/reference:

  merge_lora_into_weight   utils/convert_edlora_to_diffusers.py:36-81   (module imports only `copy`: loaded as a file)
  select_frame_idx         data/frame_point_dataset.py:13-22            } their modules import PIL / torchvision / CLIP, so the
  bind_concept_prompt      utils/edlora_util.py:100-111                 } single function is compiled from the file's AST
                                                                          (executed from /root/reference, nothing is copied)

The UNet state dict is the seeded tiny configuration of the CPU tests (re-created from its seed by the test, not stored); the
fixture stores the LoRA, and for the merged result the touched tensors of a few named keys plus a digest over all of them.
A second fixture, tests/golden/edlora_merge_pair.pt, holds merge_lora_into_weight's result for two full-size weights (a
Linear and a 1x1 conv, inputs re-created from their seed by the test): every MERGE_STRIDE-th element of each merged tensor
and its float64 sum and sum of squares (the whole tensors would exceed 1 MB).
    python -m oracle.make_golden_formats"""
import ast
import hashlib
import importlib.util
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
OUT = os.path.join(ROOT, "tests", "golden", "formats.pt")
MERGE_OUT = os.path.join(ROOT, "tests", "golden", "edlora_merge_pair.pt")
REF = os.environ.get("VIDEOSWAP_REFERENCE", "/root/reference")

TINY = dict(boc=(32, 64, 128, 128), ctx=64, groups=8)
RANK, ALPHA = 4, 0.6
MERGE_STRIDE = 61


def function_from_file(path, name, env=None):
    tree = ast.parse(open(path).read())
    node = next(n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == name)
    mod = ast.Module(body=[node], type_ignores=[])
    ns = dict(env or {})
    exec(compile(mod, path, "exec"), ns)
    return ns[name]


def tiny_state_dict(dtype):
    from videoswap_b200.spec import UNetConfig, unet_param_shapes
    from videoswap_b200.weights import seeded_state_dict
    cfg = UNetConfig(block_out_channels=TINY["boc"], cross_attention_dim=TINY["ctx"], norm_num_groups=TINY["groups"])
    sd = seeded_state_dict(unet_param_shapes(cfg), seed=0)
    return {k: v.to(dtype) for k, v in sd.items()}


def make_lora(sd, seed=11):
    """LoRA pairs for every fifth matching weight (all eight site kinds, 1x1-conv and Linear, spatial and motion keys)."""
    from videoswap_b200.formats import lora_down_name
    g = torch.Generator().manual_seed(seed)
    lora, n = {}, 0
    for k, w in sd.items():
        dn = lora_down_name(k)
        if dn == k:
            continue
        n += 1
        if n % 5:
            continue
        out_f, in_f = w.shape[0], w.shape[1]
        down = 0.3 * torch.randn((RANK, in_f), generator=g)
        up = 0.3 * torch.randn((out_f, RANK), generator=g)
        if w.dim() == 4:                                   # LoRA of a 1x1 conv is stored as conv weights
            down, up = down[:, :, None, None], up[:, :, None, None]
        lora[dn], lora[dn.replace("lora_down", "lora_up")] = down, up
    lora["text_model.not_a_unet_key.lora_down.weight"] = torch.zeros(RANK, 8)      # a stray pair: ignored by the reference
    lora["text_model.not_a_unet_key.lora_up.weight"] = torch.zeros(8, RANK)
    return lora


def digest(sd, keys):
    h = hashlib.sha256()
    for k in sorted(keys):
        h.update(k.encode())
        h.update(sd[k].detach().contiguous().cpu().numpy().tobytes())
    return h.hexdigest()


def merge_pair_inputs(seed=7):
    """Two weights of the full UNet, a Linear and a 1x1 conv, with rank-4 LoRA pairs (base, lora)."""
    k1 = "down_blocks.0.attentions.0.transformer_blocks.0.attn2.to_k.weight"
    k2 = "down_blocks.0.attentions.0.proj_in.weight"                       # 4-D 1x1 conv weight
    g = torch.Generator().manual_seed(seed)
    base = {k1: torch.randn((320, 768), generator=g), k2: torch.randn((320, 320, 1, 1), generator=g)}
    lora = {k1.replace("to_k.weight", "to_k.lora_down.weight"): torch.randn((RANK, 768), generator=g),
            k1.replace("to_k.weight", "to_k.lora_up.weight"): torch.randn((320, RANK), generator=g),
            k2.replace("proj_in.weight", "proj_in.lora_down.weight"): torch.randn((RANK, 320, 1, 1), generator=g),
            k2.replace("proj_in.weight", "proj_in.lora_up.weight"): torch.randn((320, RANK, 1, 1), generator=g)}
    return base, lora


def merge_pair_summary(merged):
    """What edlora_merge_pair.pt keeps of a merged tensor."""
    flat = merged.reshape(-1)
    return {"shape": tuple(merged.shape), "sample": flat[::MERGE_STRIDE].clone(),
            "sum": float(flat.double().sum()), "sumsq": float((flat.double() ** 2).sum())}


def reference_convert():
    spec = importlib.util.spec_from_file_location("ref_convert_edlora", os.path.join(REF, "videoswap/utils/convert_edlora_to_diffusers.py"))
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    return ref


def write_merge_pair(ref):
    base, lora = merge_pair_inputs()
    merged = ref.merge_lora_into_weight(base, lora, model_type="unet", alpha=ALPHA)
    torch.save({"alpha": ALPHA, "stride": MERGE_STRIDE, "merged": {k: merge_pair_summary(merged[k]) for k in base}}, MERGE_OUT)
    print("wrote", MERGE_OUT, os.path.getsize(MERGE_OUT), "bytes")


def main():
    ref = reference_convert()
    write_merge_pair(ref)
    select_frame_idx = function_from_file(os.path.join(REF, "videoswap/data/frame_point_dataset.py"), "select_frame_idx")
    bind_concept_prompt = function_from_file(os.path.join(REF, "videoswap/utils/edlora_util.py"), "bind_concept_prompt")

    out = {"alpha": ALPHA, "rank": RANK, "tiny": TINY}
    lora = make_lora(tiny_state_dict(torch.float32))
    out["lora"] = {k: v.clone() for k, v in lora.items()}
    for tag, dtype in (("fp32", torch.float32), ("fp16", torch.float16)):
        sd = tiny_state_dict(dtype)
        merged = ref.merge_lora_into_weight(sd, lora, model_type="unet", alpha=ALPHA)
        touched = [k for k in sd if not torch.equal(merged[k].to(torch.float32), sd[k].to(torch.float32)) or merged[k].dtype != sd[k].dtype]
        # what load_state_dict into parameters of `dtype` leaves behind (one rounding)
        final = {k: merged[k].to(dtype) for k in touched}
        sample = sorted(touched)[:: max(1, len(touched) // 10)]
        out[tag] = {"touched": sorted(touched), "digest": digest(final, touched), "sample": {k: final[k].clone() for k in sample}}
        print(tag, "touched", len(touched), "sample", len(sample))

    out["select_frame_idx"] = [((b, e, n), select_frame_idx(b, e, n)) for b, e, n in
                               ((0, 16, 16), (0, 32, 16), (0, 60, 16), (0, 100, 8), (3, 50, 16), (0, 15, 16), (0, 31, 16), (0, 200, 32))]
    cfg = {"<new1>": {"concept_token_names": [f"<new1_{i}>" for i in range(16)], "concept_token_ids": list(range(16))},
           "<new2>": {"concept_token_names": [f"<new2_{i}>" for i in range(16)], "concept_token_ids": list(range(16, 32))}}
    cfg1 = {"<new1>": {"concept_token_names": ["<new1_0>"], "concept_token_ids": [0]}}
    prompts = ["a <new1> walking", ["a <new1> next to a <new2>", "no concept here"]]
    out["bind"] = [(p, c, bind_concept_prompt(p, c)) for p in prompts for c in (cfg, cfg1)]
    torch.save(out, OUT)
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
