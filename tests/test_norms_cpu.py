"""CPU: the fused-norm entry points' argument validation, the module selection of ``install_fused_norms`` on the SDXL and
tiny fixtures, and the absence of a CPU fallback."""
import ctypes as C

import pytest
import torch

from fixtures import sdxl_unet


def test_struct_ids_and_workspace_query(built_lib):
    from pairwise_sample_optimization_b200 import _lib
    lib = _lib.lib()  # raises on a struct-size mismatch
    assert lib.psob200_struct_size(14) == C.sizeof(_lib.LayerNormArgs)
    assert lib.psob200_struct_size(15) == C.sizeof(_lib.GroupNormArgs)
    # 8 samples x 32 groups of a 960-channel 128x128 map: 30 x 16384 elements per group, 60 parts of 8192, 8 bytes each
    assert lib.psob200_group_norm_workspace_bytes(8, 960, 128 * 128, 32) == 8 * 32 * 60 * 8
    assert lib.psob200_group_norm_workspace_bytes(1, 4, 63, 4) == 4 * 8
    assert lib.psob200_group_norm_workspace_bytes(1, 30, 64, 32) == 0  # C not divisible by G


def test_layer_norm_validation(built_lib):
    from pairwise_sample_optimization_b200 import _lib
    lib = _lib.lib()
    assert lib.psob200_layer_norm_forward(None, None) == -1 and lib.psob200_layer_norm_backward(None, None) == -1
    a = _lib.LayerNormArgs()
    a.x, a.y, a.mean, a.rstd, a.rows, a.C, a.ld_x, a.ld_y = 256, 512, 1024, 2048, 4, 640, 640, 640
    a.dtype, a.out_dtype, a.param_dtype = _lib.BF16, _lib.BF16, _lib.BF16
    a.rows = 0
    assert lib.psob200_layer_norm_forward(C.byref(a), None) == -1  # no rows
    a.rows = 4
    assert lib.psob200_layer_norm_backward(C.byref(a), None) == -1  # no dy / dx
    a.out_dtype = _lib.F16
    assert lib.psob200_layer_norm_forward(C.byref(a), None) == -2  # output neither the input type nor fp32
    a.out_dtype = _lib.BF16
    a.C, a.ld_x, a.ld_y = 636, 636, 636
    assert lib.psob200_layer_norm_forward(C.byref(a), None) == -5  # row width not a multiple of 8
    a.C, a.ld_x, a.ld_y = 4096, 4096, 4096
    assert lib.psob200_layer_norm_forward(C.byref(a), None) == -5  # wider than 2048
    a.C, a.ld_x, a.ld_y, a.x = 640, 640, 640, 264
    assert lib.psob200_layer_norm_forward(C.byref(a), None) == -3  # misaligned input


def test_group_norm_validation(built_lib):
    from pairwise_sample_optimization_b200 import _lib
    lib = _lib.lib()
    assert lib.psob200_group_norm_forward(None, None) == -1 and lib.psob200_group_norm_backward(None, None) == -1
    a = _lib.GroupNormArgs()
    a.x, a.y, a.mean, a.rstd, a.workspace, a.workspace_bytes = 256, 512, 1024, 2048, 4096, 16
    a.N, a.C, a.HW, a.G = 2, 64, 49, 32
    a.dtype, a.out_dtype, a.param_dtype = _lib.F16, _lib.F32, _lib.F32
    a.workspace = None
    assert lib.psob200_group_norm_forward(C.byref(a), None) == -1  # no workspace
    a.workspace = 4096
    a.param_dtype = 7
    assert lib.psob200_group_norm_forward(C.byref(a), None) == -2
    a.param_dtype, a.C = _lib.F32, 60
    assert lib.psob200_group_norm_forward(C.byref(a), None) == -5  # C not divisible by G
    a.C, a.y = 64, 520
    assert lib.psob200_group_norm_forward(C.byref(a), None) == -3  # misaligned output
    a.y = 512
    assert lib.psob200_group_norm_forward(C.byref(a), None) == -6  # 2 x 32 parts need 512 bytes of workspace


def _counts(cfg, device):
    from pairwise_sample_optimization_b200 import norms
    with torch.device(device):
        unet = sdxl_unet.UNet2DConditionModel(cfg)
    return norms.install_fused_norms(unet)


def test_install_counts_sdxl_on_meta():
    # SDXL: 70 transformer blocks x 3 LayerNorms; 17 ResNet blocks x 2 + 11 Transformer2DModel + conv_norm_out GroupNorms
    assert _counts(sdxl_unet.sdxl_config(), "meta") == {"layer_norm": 210, "group_norm": 46, "resnet_block": 17}


def test_install_counts_tiny():
    assert _counts(sdxl_unet.tiny_config(), "cpu") == {"layer_norm": 36, "group_norm": 31, "resnet_block": 12}


def test_install_skips_what_the_kernels_do_not_take():
    from pairwise_sample_optimization_b200 import norms
    model = torch.nn.ModuleList([torch.nn.LayerNorm(36), torch.nn.LayerNorm((8, 8)), torch.nn.LayerNorm(4096),
                                 torch.nn.LayerNorm(64)])
    assert norms.install_fused_norms(model) == {"layer_norm": 1, "group_norm": 0, "resnet_block": 0}
    assert "forward" in vars(model[3]) and "forward" not in vars(model[0])

    class ResnetBlock2D(torch.nn.Module):  # diffusers' class with a non-default configuration is left alone
        def __init__(self, **cfg):
            super().__init__()
            self.norm1, self.norm2 = torch.nn.GroupNorm(4, 8), torch.nn.GroupNorm(4, 8)
            self.conv1 = self.conv2 = torch.nn.Conv2d(8, 8, 1)
            self.time_emb_proj, self.conv_shortcut = torch.nn.Linear(8, 8), None
            self.nonlinearity, self.dropout = torch.nn.SiLU(), torch.nn.Dropout(0.0)
            self.upsample = self.downsample = None
            self.time_embedding_norm, self.output_scale_factor, self.skip_time_act = "default", 1.0, False
            for k, v in cfg.items():
                setattr(self, k, v)

    for cfg, want in (({}, 1), ({"time_embedding_norm": "scale_shift"}, 0), ({"output_scale_factor": 2.0}, 0),
                      ({"skip_time_act": True}, 0), ({"dropout": torch.nn.Dropout(0.1)}, 0),
                      ({"downsample": torch.nn.Identity()}, 0), ({"nonlinearity": torch.nn.Mish()}, 0)):
        assert norms.install_fused_norms(ResnetBlock2D(**cfg))["resnet_block"] == want, cfg


def test_cpu_tensors_raise(built_lib):
    from pairwise_sample_optimization_b200 import _lib, norms
    with pytest.raises(_lib.Psob200Error, match="CUDA"):
        norms.layer_norm(torch.randn(4, 64), torch.ones(64), torch.zeros(64))
    with pytest.raises(_lib.Psob200Error, match="CUDA"):
        norms.group_norm(torch.randn(2, 8, 4, 4), 4, silu=True, channel_add=torch.randn(2, 8))
    with pytest.raises(_lib.Psob200Error, match="gradient"):
        norms.layer_norm(torch.randn(4, 64), torch.ones(64, requires_grad=True))
