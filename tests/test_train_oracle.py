"""The oracle's training step (autograd over the functional restatement, train-mode BatchNorm, Focal-R) is pinned to
the REAL reference: tests/golden/metnet3_small128_train.pt was produced by tests/golden/make_golden.py from
/root/reference/src/metnet3.py in train() mode (dropout 0) and holds the loss, the prediction and, per parameter,
the gradient norm and 48 sampled gradient entries."""
import torch

from oracle import synth
from oracle.focal_r_oracle import focal_r
from oracle.metnet3_oracle import metnet3_forward


def oracle_train_step(cfg, B, wseed, iseed):
    sd = synth.make_state_dict(synth.metnet3_spec(cfg), seed=wseed)
    for k, v in sd.items():
        if v.is_floating_point() and "running_" not in k and k != "pm25_boundaries":
            v.requires_grad_(True)
    x, ts, target = synth.make_inputs(cfg, B, seed=iseed)
    pred = metnet3_forward(x, ts, sd, cfg, training=True)
    loss = focal_r(pred, target)
    loss.backward()
    return sd, pred.detach(), loss.detach()


def test_oracle_training_step_matches_reference(golden):
    f = golden("metnet3_small128_train.pt")
    cfg = synth.GridConfig(**f["cfg"])
    # the fixture was generated with 8 torch CPU threads (make_golden.py).  The float32 reduction order of the CPU
    # backward follows the thread count, and the sampled-gradient error moves with it (7.8e-4 at 1 to 4 threads, 1.3e-4
    # at 16, 8.5e-5 at 8 on the same inputs), so the oracle runs with the fixture's thread count on any host.
    threads = torch.get_num_threads()
    torch.set_num_threads(8)
    try:
        sd, pred, loss = oracle_train_step(cfg, f["B"], f["weight_seed"], f["input_seed"])
    finally:
        torch.set_num_threads(threads)
    assert abs(loss.item() - f["loss"]) < 1e-5 * abs(f["loss"])
    assert ((pred - f["pred"]).abs().max() / f["pred"].abs().max()).item() < 1e-4
    assert set(f["grads"]) == {k for k, v in sd.items() if v.requires_grad}
    worst = 0.0
    for k, g in f["grads"].items():
        got = sd[k].grad.reshape(-1)
        # conv biases in front of a batch-statistic BatchNorm have an analytically zero gradient (float noise ~1e-6
        # against norms of 0.15 .. 140 elsewhere): absolute floor 1e-4
        assert abs(got.norm().item() - g["norm"]) <= 1e-3 * g["norm"] + 1e-4, k
        err = (got[g["idx"]] - g["val"]).abs().max().item() / max(g["absmax"], 1e-2)
        worst = max(worst, err)
    assert worst < 1e-4, worst
