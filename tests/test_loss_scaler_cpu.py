"""CPU: the device loss scaler's host side -- the NumPy restatement of the scale update against torch's own
``torch._amp_update_scale_``, the C ABI of the four ``*_scaled`` entry points (struct size, argument checks made before any
CUDA call) and ``DeviceGradScaler``'s state in torch's ``GradScaler`` format."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import loss_scaler as ols


@pytest.mark.parametrize("growth,backoff,interval", [(2.0, 0.5, 3), (1.3, 0.7, 2), (2.0, 0.5, 1), (1.0001, 0.9999, 5)])
def test_update_rule_matches_torch(growth, backoff, interval):
    """Random overflow patterns over many updates, power-of-two and other factors: scale and tracker equal torch's."""
    rng = np.random.default_rng(interval)
    for init in (2.0 ** 16, 3.0e38, 1.1e-38, 7.0):
        scale_t = torch.full((1,), init, dtype=torch.float32)
        tracker_t = torch.zeros(1, dtype=torch.int32)
        scale, tracker = np.float32(init), 0
        for found in rng.random(200) < 0.2:
            torch._amp_update_scale_(scale_t, tracker_t, torch.full((1,), float(found)), growth, backoff, interval)
            scale, tracker = ols.update_scale(scale, tracker, bool(found), growth, backoff, interval)
            assert scale_t.numpy()[0].tobytes() == np.float32(scale).tobytes() and int(tracker_t) == tracker


def test_growth_stops_at_the_fp32_range():
    scale, tracker = ols.update_scale(np.float32(3.0e38), 0, False, 2.0, 0.5, 1)
    assert scale == np.float32(3.0e38) and tracker == 0
    assert ols.unscale_factor(np.float32(2.0 ** 16)) == np.float32(2.0 ** -16)
    assert ols.unscale_factor(np.float32(3.0)) == np.float32(1.0 / 3.0)


def test_struct_size_matches_the_ctypes_mirror(built_lib):
    from pairwise_sample_optimization_b200 import _lib
    lib = _lib.lib()
    assert lib.psob200_struct_size(13) == C.sizeof(_lib.LossScaler) == 40
    assert lib.psob200_abi_version() == 2


def _scaler(**kw):
    from pairwise_sample_optimization_b200 import _lib
    s = _lib.LossScaler()
    s.scale, s.growth_tracker, s.growth_factor, s.backoff_factor, s.growth_interval = 4096, 4352, 2.0, 0.5, 2000
    for k, v in kw.items():
        setattr(s, k, v)
    return s


def test_scaled_entry_points_check_the_scaler_before_any_cuda_call(built_lib):
    """Every argument would otherwise reach a launch (valid pointers are fake): the checks must return first."""
    from pairwise_sample_optimization_b200 import _lib
    lib = _lib.lib()
    sched = _lib.Schedule()
    sched.kind = _lib.SCHED_AFFINE
    on = _lib.OnlinePsoArgs()
    db = _lib.DreamboothArgs()
    o32 = _lib.FlatAdamwArgs()
    o32.param = o32.grad = o32.exp_avg = o32.exp_avg_sq = o32.workspace = 4096
    o32.n, o32.step = 8, 1
    o8 = _lib.FlatAdamw8Args()
    o8.param = o8.grad = o8.workspace = o8.code1 = o8.code2 = o8.absmax1 = o8.absmax2 = o8.map1 = o8.map2 = o8.blocks8 = 4096
    o8.n, o8.step, o8.n_blocks8, o8.block_size = 4096, 1, 16, 256
    loss_calls = (lambda s: lib.psob200_online_pso_loss_grad_scaled(C.byref(sched), C.byref(on), s, None),
                  lambda s: lib.psob200_dreambooth_pso_loss_grad_scaled(C.byref(db), s, None))
    opt_calls = (lambda s: lib.psob200_flat_adamw_step_scaled(C.byref(o32), s, None),
                 lambda s: lib.psob200_flat_adamw8_step_scaled(C.byref(o8), s, None))
    for call in loss_calls + opt_calls:
        assert call(None) == -1                              # no scaler
        assert call(C.byref(_scaler(scale=None))) == -1      # no scale
    for call in opt_calls:
        for bad in (dict(growth_tracker=None), dict(growth_interval=0), dict(growth_interval=-3), dict(growth_factor=1.0),
                    dict(growth_factor=0.5), dict(growth_factor=float("nan")), dict(backoff_factor=0.0),
                    dict(backoff_factor=1.0), dict(backoff_factor=-0.5), dict(backoff_factor=float("nan"))):
            assert call(C.byref(_scaler(**bad))) == -1, bad
    # the loss entry points read only the scale: a scaler without a tracker is accepted there (and then the loss's own
    # argument checks answer: B = 0 / NULL pointers)
    assert lib.psob200_online_pso_loss_grad_scaled(C.byref(sched), C.byref(on), C.byref(_scaler(growth_tracker=None)),
                                                   None) == -1
    assert lib.psob200_online_pso_loss_grad_scaled(None, None, C.byref(_scaler()), None) == -1
    assert lib.psob200_flat_adamw_step_scaled(None, C.byref(_scaler()), None) == -1
    o32.n_sumsq_parts = 2  # the unscaled boundary's own checks still apply behind a valid scaler
    assert lib.psob200_flat_adamw_step_scaled(C.byref(o32), C.byref(_scaler()), None) == -1
    o8.block_size = 512
    assert lib.psob200_flat_adamw8_step_scaled(C.byref(o8), C.byref(_scaler()), None) == -5


def test_device_grad_scaler_round_trips_torch_state():
    from pairwise_sample_optimization_b200 import amp
    ts = torch.amp.GradScaler("cpu", init_scale=1024.0, growth_factor=1.5, backoff_factor=0.25, growth_interval=7)
    sd = ts.state_dict()
    assert set(sd) == {"scale", "growth_factor", "backoff_factor", "growth_interval", "_growth_tracker"}
    ds = amp.DeviceGradScaler("cpu")
    ds.load_state_dict(sd)
    assert ds.state_dict() == sd
    assert ds.get_scale() == 1024.0 and ds.scale_tensor.dtype == torch.float32 and ds.growth_tracker.dtype == torch.int32
    # a state with a grown tracker and a non-power-of-two scale, and back into torch
    sd2 = dict(sd, scale=3000.5, _growth_tracker=5)
    ds.load_state_dict(sd2)
    assert ds.state_dict() == sd2
    ts2 = torch.amp.GradScaler("cpu")
    ts2.load_state_dict(ds.state_dict())
    assert ts2.state_dict() == sd2
    # defaults are torch's
    d0, t0 = amp.DeviceGradScaler("cpu").state_dict(), torch.amp.GradScaler("cpu").state_dict()
    assert d0 == t0
    loss = torch.tensor(0.75)
    assert ds.scale(loss).item() == 0.75 * 3000.5
    with pytest.raises(RuntimeError, match="empty"):
        ds.load_state_dict({})
    for bad in (dict(growth_factor=1.0), dict(backoff_factor=1.0), dict(growth_interval=0)):
        with pytest.raises(ValueError):
            amp.DeviceGradScaler("cpu", **bad)


def test_kernel_paths_refuse_a_scaler_that_is_not_on_the_device():
    from pairwise_sample_optimization_b200 import _lib, amp
    with pytest.raises(_lib.Psob200Error, match="DeviceGradScaler"):
        amp.scaler_arg(torch.amp.GradScaler("cpu"), torch.device("cuda", 0))
    with pytest.raises(_lib.Psob200Error, match="lives on"):
        amp.scaler_arg(amp.DeviceGradScaler("cpu"), torch.device("cuda", 0))
