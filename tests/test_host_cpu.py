"""CPU tests (no GPU): the C-ABI library loads and exports every declared symbol, the host-side mirror has the
reference's module tree / state_dict keys, scheduler tables match the oracle, failure modes are loud, and the product
package never imports the oracle."""
import os
import re

import pytest
import torch

import videoswap_b200 as V
from oracle import unet3d_oracle as O
from videoswap_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_loads_and_exports_every_header_symbol():
    lib = _lib.lib()
    syms = _lib.header_symbols()
    assert len(syms) >= 25
    missing = [s for s in syms if not hasattr(lib, s)]
    assert not missing, missing
    assert set(syms) == set(_lib._SIGNATURES), set(syms) ^ set(_lib._SIGNATURES)
    assert lib.vs_version() >= 100


def test_model_tree_matches_reference_surface():
    m = V.AnimateDiffUNet3DModel(init="empty")
    sd = m.state_dict()
    shapes = V.unet_param_shapes(m.cfg)
    assert {k: tuple(v.shape) for k, v in sd.items()} == dict(shapes)
    n_params = sum(v.numel() for k, v in sd.items() if not k.endswith(".pe"))
    assert n_params == 1_276_658_564            # 859.5 M SD-1.5 + 417.1 M motion modules (SURVEY 0.4)
    # the walk of revise_edlora_unet_attention_forward (edlora_util.py:85-99): class name 'Attention', 'attn2' in name
    count = 0

    def walk(mod):
        nonlocal count
        for name, layer in mod.named_children():
            if layer.__class__.__name__ == "Attention" and "attn2" in name:
                layer.set_processor(object())
                count += 1
            else:
                walk(layer)
    walk(m.down_blocks), walk(m.mid_block), walk(m.up_blocks)
    assert count == 16
    assert sum(1 for k, _ in m.named_modules() if k.endswith("temporal_transformer")) == 20
    assert m.config.in_channels == 4 and m.config.sample_size == 64
    a = m.down_blocks[0].attentions[0].transformer_blocks[0].attn1
    assert a.heads == 8 and abs(a.scale - 40 ** -0.5) < 1e-9 and a.to_q.weight.shape == (320, 320)
    assert "down_blocks.0.motion_modules.0.temporal_transformer.transformer_blocks.0.attention_blocks.0.processor.pos_encoder.pe" in sd


def test_cpu_tensor_is_rejected_loudly():
    m = V.AnimateDiffUNet3DModel(block_out_channels=(320, 640, 1280, 1280), init="empty")
    with pytest.raises(RuntimeError, match="CUDA only"):
        m(torch.zeros(1, 4, 1, 8, 8), 1, torch.zeros(1, 77, 768))


def test_missing_library_is_an_error(monkeypatch):
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libvideoswap_b200.so")
    with pytest.raises(_lib.VSError, match="no CPU/PyTorch fallback"):
        _lib.lib()


def test_scheduler_tables_match_oracle():
    s = V.DDIMScheduler()
    s.set_timesteps(50)
    o = O.DDIM()
    assert s.timesteps == o.timesteps(50)
    assert torch.allclose(s.alphas_cumprod, o.alphas_cumprod)
    a_t, a_p = s.alphas(981)
    assert abs(a_t - float(o.alphas_cumprod[981])) < 1e-9 and abs(a_p - float(o.alphas_cumprod[961])) < 1e-9
    a_t, a_p = s.alphas(1)
    assert abs(a_p - float(o.alphas_cumprod[0])) < 1e-9       # set_alpha_to_one=False
    inv = V.DDIMInverseScheduler()
    inv.set_timesteps(50)
    assert inv.timesteps == o.inverse_timesteps(50)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "videoswap_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f
                assert "/root/reference" not in text, f


def test_bench_dump_outputs_float32_and_seeded_sample(tmp_path):
    """bench.py --dump-outputs: float32 .npy files; over the byte limit, the same sorted sample positions every run."""
    import numpy as np
    import bench
    x = torch.arange(4 * 16, dtype=torch.float16).reshape(4, 16)
    bench.dump_outputs(str(tmp_path / "full"), {"latents": x})
    a = np.load(tmp_path / "full" / "latents.npy")
    assert a.dtype == np.float32 and a.shape == (4, 16) and np.array_equal(a, x.float().numpy())
    for run in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / run), {"latents": x, "eps": 2 * x}, limit=128)
    s1, s2 = np.load(tmp_path / "s1" / "latents.npy"), np.load(tmp_path / "s2" / "latents.npy")
    assert s1.dtype == np.float32 and s1.size == 16 and np.array_equal(s1, s2)
    assert np.all(np.diff(s1) > 0) and set(s1.tolist()) <= set(range(64))       # sorted positions of arange = values
    assert np.array_equal(np.load(tmp_path / "s1" / "eps.npy"), 2 * s1)           # every array sampled at the same positions


def test_registry_names():
    assert V.build_model("AnimateDiffUNet3DModel") is V.AnimateDiffUNet3DModel
    assert V.build_model("UNet3DConditionModel") is V.AnimateDiffUNet3DModel
    assert V.build_pipeline("TuneAVideoPipeline") is V.VideoSwapPipeline


def test_layernorm_folding_algebra():
    """LN(x)(+pe) W^T + b == rstd (x W'^T) - rstd mean u + c (+ cpe): the identity behind ln_fold / EPI_F_LN (gemm.cu)."""
    import torch
    g = torch.Generator().manual_seed(5)
    rows, C, N, F, hw = 60, 320, 96, 3, 4
    x = torch.randn(rows, C, generator=g, dtype=torch.float64) * 2 + 0.7
    gamma = 1 + 0.1 * torch.randn(C, generator=g, dtype=torch.float64)
    beta = 0.1 * torch.randn(C, generator=g, dtype=torch.float64)
    W = torch.randn(N, C, generator=g, dtype=torch.float64) / C ** 0.5
    b = torch.randn(N, generator=g, dtype=torch.float64)
    pe = torch.randn(F, C, generator=g, dtype=torch.float64)
    frame = (torch.arange(rows) // hw) % F
    ref = (torch.nn.functional.layer_norm(x, (C,), gamma, beta, 1e-5) + pe[frame]) @ W.t() + b
    mean = x.mean(1, keepdim=True)
    rstd = (x.var(1, unbiased=False, keepdim=True) + 1e-5).rsqrt()
    Wf = W * gamma                       # folded weights
    u = Wf.sum(1)                        # row sums
    c = W @ beta + b                     # constant offset
    cpe = pe @ W.t()                     # per-frame positional offsets
    out = rstd * (x @ Wf.t()) + (-mean * rstd) * u + c + cpe[frame]
    assert torch.allclose(out, ref, atol=1e-9)


def test_from_pretrained_2d_contract(tmp_path):
    """The reference builds the model with from_pretrained_2d(path, subfolder='unet', unet_additional_kwargs=...) from a
    2-D SD checkpoint (unet.py:483-523, test.py:52-58): config.json keys it does not know are ignored, the 2-D weights
    load with strict=False and the motion-module parameters are the missing keys."""
    import json
    import torch
    cfg2d = {"_class_name": "UNet2DConditionModel", "_diffusers_version": "0.6.0", "act_fn": "silu", "attention_head_dim": 8,
             "block_out_channels": [320, 640, 1280, 1280], "center_input_sample": False, "cross_attention_dim": 768,
             "down_block_types": ["CrossAttnDownBlock2D"] * 3 + ["DownBlock2D"], "downsample_padding": 1,
             "flip_sin_to_cos": True, "freq_shift": 0, "in_channels": 4, "layers_per_block": 2, "mid_block_scale_factor": 1,
             "norm_eps": 1e-05, "norm_num_groups": 32, "out_channels": 4, "sample_size": 64,
             "up_block_types": ["UpBlock2D"] + ["CrossAttnUpBlock2D"] * 3}
    d = tmp_path / "sd" / "unet"
    d.mkdir(parents=True)
    (d / "config.json").write_text(json.dumps(cfg2d))
    shapes = V.unet_param_shapes(V.UNetConfig())
    # a PARTIAL 2-D checkpoint (biases / norm parameters only: no 3 GB file); strict=False must accept it
    ckpt = {k: torch.zeros(v) for k, v in shapes.items() if "motion_modules" not in k and len(v) == 1}
    ckpt["conv_in.bias"] = torch.full((320,), 0.25)
    torch.save(ckpt, d / "diffusion_pytorch_model.bin")
    kw = {"use_motion_module": True, "motion_module_type": "Vanilla",
          "motion_module_kwargs": {"num_attention_heads": 8, "num_transformer_block": 1,
                                   "attention_block_types": ["Temporal_Self", "Temporal_Self"],
                                   "temporal_position_encoding": True, "temporal_position_encoding_max_len": 24}}
    m = V.AnimateDiffUNet3DModel.from_pretrained_2d(str(tmp_path / "sd"), subfolder="unet", unet_additional_kwargs=kw)
    assert isinstance(m, V.AnimateDiffUNet3DModel)
    assert torch.allclose(m.conv_in.bias.float(), torch.full((320,), 0.25))            # loaded
    assert sum(1 for k in m.state_dict() if "motion_modules" in k) == 560              # present, left at their init
    # ... and that init is the reference's: every temporal_transformer.proj_out is ZERO (motion_module.py:76-77), so a
    # motion module is an exact identity until a motion checkpoint arrives (ADVICE r1); other motion weights are not zero
    po = [v for k, v in m.state_dict().items() if ".temporal_transformer.proj_out." in k]
    assert len(po) == 40 and all(float(v.abs().max()) == 0.0 for v in po)
    assert float(m.state_dict()["down_blocks.0.motion_modules.0.temporal_transformer.proj_in.weight"].abs().max()) > 0
    with pytest.raises(RuntimeError):
        V.AnimateDiffUNet3DModel.from_pretrained_2d(str(tmp_path / "nope"), subfolder="unet")


def test_inverse_scheduler_conventions_and_alpha_table():
    """DDIM / inverse-DDIM index arithmetic against an independent float64 restatement of the SD-1.5 schedule
    (scaled_linear 0.00085 -> 0.012, 1000 steps), for all 50 steps of both DDIMInverseScheduler conventions (ADVICE r1)."""
    import numpy as np
    betas = np.linspace(0.00085 ** 0.5, 0.012 ** 0.5, 1000, dtype=np.float64) ** 2
    ac = np.cumprod(1.0 - betas)
    fwd = V.DDIMScheduler()
    fwd.set_timesteps(50)
    assert fwd.timesteps == [981 - 20 * i for i in range(50)]
    for t in fwd.timesteps:
        a_t, a_p = fwd.alphas(t)
        assert abs(a_t - ac[t]) < 2e-6 and abs(a_p - (ac[t - 20] if t >= 20 else ac[0])) < 2e-6
    old = V.DDIMInverseScheduler(convention="0.19.3")
    new = V.DDIMInverseScheduler(convention="0.21")
    assert V.DDIMInverseScheduler().convention == "0.19.3"        # the release the reference pins (requirements.txt:2)
    for s_ in (old, new):
        s_.set_timesteps(50)
        assert s_.timesteps == [1 + 20 * i for i in range(50)]
    for t in old.timesteps:      # UNet at t, x0 from alpha[t], moves to alpha[t + 20] (alphas_cumprod[-1] beyond the table)
        a_cur, a_nxt = old.alphas(t)
        assert abs(a_cur - ac[t]) < 2e-6 and abs(a_nxt - (ac[t + 20] if t + 20 < 1000 else ac[999])) < 2e-6
        assert a_nxt < a_cur                                         # noise level increases
    for t in new.timesteps:      # UNet at the target t, sample at t - 20 (alphas_cumprod[0] before the table)
        a_cur, a_nxt = new.alphas(t)
        assert abs(a_nxt - ac[t]) < 2e-6 and abs(a_cur - (ac[t - 20] if t >= 20 else ac[0])) < 2e-6
    with pytest.raises(ValueError):
        V.DDIMInverseScheduler(convention="0.20")


def test_attention_control_registration_and_store_protocol():
    """SURVEY 8f-2, host side: register_attention_control walks attn1 / attn2 like the reference
    (attention_register.py:176-211: 16 + 16 layers, ED-LoRA index on the cross layers), and the device-agnostic part of the
    store follows attention_store.py (only the conditional half under CFG, running sum, per-step list)."""
    from videoswap_b200 import p2p
    m = V.AnimateDiffUNet3DModel(init="empty")
    ctl = p2p.AttentionStore()
    assert p2p.register_attention_control(m, ctl) == 32 and ctl.num_att_layers == 32
    a2 = m.up_blocks[1].attentions[0].transformer_blocks[0].attn2.processor
    assert isinstance(a2, p2p.EDLoRA_AttnControlProcessor) and a2.place_in_unet == "up" and a2.controller is ctl
    assert a2.cross_attention_idx == 7                       # 6 down + 1 mid before the first up transformer
    assert m._check_processors() is ctl
    p2p.register_attention_control(m, None)
    assert m._check_processors() is None
    # store protocol on plain tensors
    ctl = p2p.AttentionStore()
    for step in range(2):
        for place, cross in (("down", False), ("down", True), ("up", True)):
            attn = torch.full((4, 2, 16, 77 if cross else 16), float(step + 1))
            attn[:2] = -1.0                                  # unconditional half: must never be stored
            out = ctl(attn, cross, place)
            assert out is attn
        big = torch.zeros((4, 2, 1024, 16))
        ctl(big, False, "up")                                # >= 32^2 queries: passes through, not stored
        ctl.step_callback(torch.zeros(1, 4, 2, 8, 8))
    assert ctl.cur_step == 2 and len(ctl.attention_store_all_step) == 2 and len(ctl.latents_store) == 2
    assert [len(v) for v in ctl.attention_store.values()] == [1, 0, 1, 1, 0, 0]
    assert float(ctl.attention_store["down_cross"][0].min()) == 3.0 and ctl.attention_store["down_cross"][0].shape[0] == 2
    assert float(ctl.get_average_attention()["up_cross"][0].mean()) == 1.5
    assert float(ctl.attention_store_all_step[0]["down_self"][0].max()) == 1.0      # per-step copies are not the running sum


def test_on_disk_formats_of_the_callers_load_unchanged(tmp_path):
    """SURVEY 8f-4, the UNet-side file formats: (i) AnimateDiff motion checkpoints after test.py:63's key remap
    ('.pos_encoder' -> '.processor.pos_encoder') match our keys exactly; (ii) adapter.pth is the SparsePointAdapter
    state_dict; (iii) TAP.pth is the dict frame_point_dataset.py:66-70 turns into `conditions`; (iv) an ED-LoRA '.pth'
    ({'params': {'unet': {...lora_down / lora_up...}}}) merges through state_dict()/load_state_dict() exactly like
    convert_edlora_to_diffusers.py:70-76 (tests/golden/edlora_merge_pair.pt: the reference's own function on the same seeded
    inputs, oracle/make_golden_formats.py)."""
    m = V.AnimateDiffUNet3DModel(init="empty")
    keys = set(m.state_dict().keys())
    motion = {k for k in keys if ".motion_modules." in k}
    as_shipped = {k.replace(".processor.pos_encoder", ".pos_encoder") for k in motion}          # AnimateDiff's own naming
    remapped = {k.replace(".pos_encoder", ".processor.pos_encoder") for k in as_shipped}          # test.py:63
    assert remapped == motion and len(motion) == 560
    sd = {k: torch.zeros_like(v) for k, v in m.state_dict().items() if k in motion}
    missing, unexpected = m.load_state_dict(sd, strict=False)
    assert not unexpected and all(".motion_modules." not in k for k in missing)
    # adapter.pth / TAP.pth
    ad = V.SparsePointAdapter(init="seeded")
    torch.save(ad.state_dict(), tmp_path / "adapter.pth")
    ad2 = V.SparsePointAdapter(init="empty")
    ad2.load_state_dict(torch.load(tmp_path / "adapter.pth"))
    assert sorted(ad2.state_dict()) == sorted(f"model_list.{l}.mlp.{i}.{p}" for l in range(4) for i in (0, 2) for p in ("weight", "bias"))
    tap = {"pred_tracks": torch.rand(16, 5, 2) * 512, "point_name2id": {"nose": 0, "tail": 4}, "point_embedding": torch.randn(5, 1280)}
    torch.save(tap, tmp_path / "TAP.pth")
    t = torch.load(tmp_path / "TAP.pth")
    cond = {"pred_tracks": t["pred_tracks"], "point_embedding": t["point_embedding"], "point_name2id": t["point_name2id"],
            "img_size": (512, 512), "index_list": [t["point_name2id"]["nose"]]}
    assert cond["pred_tracks"].shape == (16, 5, 2) and cond["point_embedding"].shape[1] == 1280
    # ED-LoRA merge on two layers (rank 4), restated and compared with the reference's own function's result
    from oracle.make_golden_formats import merge_pair_inputs, merge_pair_summary
    k1 = "down_blocks.0.attentions.0.transformer_blocks.0.attn2.to_k.weight"
    k2 = "down_blocks.0.attentions.0.proj_in.weight"                       # 4-D 1x1 conv weight
    base, lora = merge_pair_inputs()
    want = {k1: base[k1] + 0.6 * lora[k1.replace("to_k.weight", "to_k.lora_up.weight")] @ lora[k1.replace("to_k.weight", "to_k.lora_down.weight")],
            k2: base[k2] + 0.6 * (lora[k2.replace("proj_in.weight", "proj_in.lora_up.weight")].squeeze() @
                                  lora[k2.replace("proj_in.weight", "proj_in.lora_down.weight")].squeeze())[..., None, None]}
    gold = torch.load(os.path.join(ROOT, "tests", "golden", "edlora_merge_pair.pt"))
    assert gold["alpha"] == 0.6 and sorted(gold["merged"]) == sorted(want)
    for k in want:
        got, ref = merge_pair_summary(want[k]), gold["merged"][k]
        assert got["shape"] == ref["shape"] and torch.allclose(got["sample"], ref["sample"], atol=1e-5), k
        assert abs(got["sum"] - ref["sum"]) <= 1e-5 * want[k].numel(), k
        assert abs(got["sumsq"] - ref["sumsq"]) <= 1e-6 * ref["sumsq"], k
    m.load_state_dict(want, strict=False)                                   # the merged dict goes back through load_state_dict
    assert torch.allclose(m.state_dict()[k1], want[k1]) and m._dirty       # ... and marks the packed weights stale
