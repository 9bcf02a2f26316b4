"""nn.SyncBatchNorm.convert_sync_batchnorm on MetNet3 and MaxViT (CPU, no kernels): the converted modules keep the state-dict
layout of the reference, so reference checkpoints -- saved from nn.DataParallel, keys prefixed 'module.' (evaluation_vit.py:
107-109) -- load into them with strict=True, and the converted BatchNorms are the ones the training path sees."""
import pytest
import torch
import torch.nn as nn

from oracle import synth


def _converted_keeps_layout(model, spec):
    before = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    conv = nn.SyncBatchNorm.convert_sync_batchnorm(model)
    assert conv is model
    after = {k: tuple(v.shape) for k, v in conv.state_dict().items()}
    assert after == before
    bns = [m for m in conv.modules() if isinstance(m, nn.modules.batchnorm._BatchNorm)]
    assert bns and all(isinstance(m, nn.SyncBatchNorm) and m.process_group is None for m in bns)
    sd = synth.make_state_dict(spec, seed=3)
    return conv, sd


@pytest.mark.parametrize("cfg", [synth.CFG_SMALL128, synth.CFG_WIDE512], ids=["small128", "wide512"])
def test_metnet3_convert_sync_batchnorm_loads_reference_checkpoint(cfg):
    from vit_grid_model_b200 import MetNet3, MetNet3_with_stn_imgs
    m, sd = _converted_keeps_layout(MetNet3(**cfg.metnet3_kwargs()), synth.metnet3_spec(cfg))
    m.load_state_dict({"module." + k: v for k, v in sd.items()}, strict=True)
    got = m.state_dict()
    assert all(torch.equal(got[k], v) for k, v in sd.items())
    # the training path's MBConv BatchNorms (train.maxvit_train_forward: seq[1], seq[4], seq[8]) are the converted modules
    for conv, _, _ in m.vit.layers:
        seq = conv.fn if hasattr(conv, "fn") else conv
        assert all(isinstance(seq[i], nn.SyncBatchNorm) for i in (1, 4, 8))
    if cfg is synth.CFG_SMALL128:
        stn_cfg = synth.CFG_STN_SMALL128
        s, sd2 = _converted_keeps_layout(MetNet3_with_stn_imgs(**stn_cfg.metnet3_kwargs()), synth.metnet3_spec(stn_cfg))
        s.load_state_dict({"module." + k: v for k, v in sd2.items()}, strict=True)


def test_tuple_depth_maxvit_convert_sync_batchnorm_loads_reference_checkpoint():
    from vit_grid_model_b200 import MaxViT
    dim, depth, heads, dh, win, R = 64, (2, 1, 1), 2, 32, 7, 4
    vit = MaxViT(dim=dim, depth=depth, cond_dim=2, heads=heads, dim_head=dh, vit_window_size=win, num_register_tokens=R)
    spec = synth.maxvit_multistage_spec(dim, depth, 2, heads, dh, win, 4, 0.25, R)
    vit, sd = _converted_keeps_layout(vit, spec)
    nn.DataParallel(vit).load_state_dict({"module." + k: v for k, v in sd.items()}, strict=True)
    got = vit.state_dict()
    assert all(torch.equal(got[k], v) for k, v in sd.items())
