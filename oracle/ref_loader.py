"""TEST INFRASTRUCTURE ONLY.  Imports the reference's OWN model files, unmodified, from a checkout of the reference
project (REFERENCE_ROOT, env VIDEOSWAP_REFERENCE) through oracle/diffusers_stub (the reference's `diffusers==0.19.3`
dependency is not installable offline).  Used by the oracle/make_golden*.py scripts that write the fixtures under
tests/golden/; no test needs the reference itself."""
import importlib
import os
import sys

REFERENCE_ROOT = os.environ.get("VIDEOSWAP_REFERENCE", "/root/reference")
_STUB = os.path.join(os.path.dirname(os.path.abspath(__file__)), "diffusers_stub")


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "videoswap", "models", "animatediff_models"))


def load_reference():
    """Returns a namespace with the reference classes (AnimateDiffUNet3DModel, SparsePointAdapter, ...)."""
    if not reference_available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    try:
        import diffusers  # noqa: F401
        if "stub" not in getattr(diffusers, "__version__", ""):
            raise RuntimeError("a real diffusers is importable; the stub must not shadow it silently")
    except ImportError:
        sys.path.insert(0, _STUB)
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    unet = importlib.import_module("videoswap.models.animatediff_models.unet")
    edlora = importlib.import_module("videoswap.utils.edlora_util")
    adapter = importlib.import_module("videoswap.models.adapter_model")

    class NS:
        AnimateDiffUNet3DModel = unet.AnimateDiffUNet3DModel
        revise_edlora_unet_attention_forward = staticmethod(edlora.revise_edlora_unet_attention_forward)
        SparsePointAdapter = adapter.SparsePointAdapter

    return NS


SD15_UNET_CONFIG = dict(  # the fields of SD-1.5's unet/config.json that the reference constructor consumes
    sample_size=64, in_channels=4, out_channels=4, center_input_sample=False, flip_sin_to_cos=True, freq_shift=0,
    block_out_channels=(320, 640, 1280, 1280), layers_per_block=2, downsample_padding=1, mid_block_scale_factor=1,
    act_fn="silu", norm_num_groups=32, norm_eps=1e-5, cross_attention_dim=768, attention_head_dim=8,
)

ADDITIONAL_KWARGS = dict(  # options/model_cfg/inference.yml:1-21 of the reference
    unet_use_cross_frame_attention=False, unet_use_temporal_attention=False, use_motion_module=True,
    motion_module_resolutions=[1, 2, 4, 8], motion_module_mid_block=False, motion_module_decoder_only=False,
    motion_module_type="Vanilla",
    motion_module_kwargs=dict(num_attention_heads=8, num_transformer_block=1,
                              attention_block_types=["Temporal_Self", "Temporal_Self"],
                              temporal_position_encoding=True, temporal_position_encoding_max_len=24,
                              temporal_attention_dim_div=1),
)


def build_reference_unet(block_out_channels=(320, 640, 1280, 1280), cross_attention_dim=768, pe_max_len=24,
                         norm_num_groups=32):
    ns = load_reference()
    cfg = dict(SD15_UNET_CONFIG, block_out_channels=tuple(block_out_channels),
               cross_attention_dim=cross_attention_dim, norm_num_groups=norm_num_groups)
    extra = dict(ADDITIONAL_KWARGS)
    extra["motion_module_kwargs"] = dict(extra["motion_module_kwargs"], temporal_position_encoding_max_len=pe_max_len)
    model = ns.AnimateDiffUNet3DModel.from_config(cfg, **extra)
    ns.revise_edlora_unet_attention_forward(model)
    return model.eval()
