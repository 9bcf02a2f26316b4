"""Synchronised BatchNorm (GPU): MaxViT BatchNorms converted with nn.SyncBatchNorm.convert_sync_batchnorm take their train-mode
statistics over the rows of every rank, so an N-rank data-parallel step is the one-GPU step on the concatenated batch.

1. The split kernels (vg_bn_stats_local / _global, vg_bn_bwd_local / _global) against float64 BatchNorm over the concatenated
   rows of three "ranks" of unequal size (one not a multiple of 256 rows, one below 256), at C = 128 .. 2048, every backward
   form (act 0 / GELU, with and without the squeeze-excite fgate / fadd), and identical bits when the global kernels run twice.
   fp32 kernel rule of DESIGN.md §2: about 1e-5 of the largest entry.
2. Two ranks on one GPU (gloo, spawned processes, both on cuda:0), a converted MetNet3 (CFG_SMALL128, dropout 0) on B = 4
   sharded 2 / 2, and a converted stand-alone MaxViT(512, heads=32, dim_head=64) (BatchNorms at hidden width 2048), in 'fp32' and
   'bf16': each rank's prediction and loss, the rank-averaged gradients and the BatchNorm running buffers against float64
   autograd through the oracle on the whole batch in train mode.  The same run without conversion fails the global-L2 check.
   Running buffers are bit-identical on both ranks; two runs under torch.use_deterministic_algorithms(True) give the same bits.
3. Unequal shards (B = 3 over two ranks): the gradients of the data-parallel objective, the mean over ranks of each rank's loss.
4. Without synchronisation nothing changes: a converted model with no process group, or with a one-rank group, gives the bits
   of the unconverted model in train() mode, eval() inference and the frozen eval() x.grad graph.
5. Two GPUs over NCCL (skipped with fewer): case 2 through DataParallel (GradSync, dedicated statistics group) and one FlatAdamW
   step; parameters and buffers are bit-identical across ranks afterwards.

Measured on a B200 (the MEASURED lines of `pytest -s`) next to each bound; bounds are at most 4x the measured value or an
existing rule of the repository."""
import io
import os
import socket
import sys

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from oracle import synth

pytestmark = pytest.mark.gpu

DEV = "cuda"
F64 = torch.float64


def note(**kv):
    print("MEASURED", " ".join(f"{k}={v:.3g}" if isinstance(v, float) else f"{k}={v}" for k, v in kv.items()))


def rel(got, ref):
    g, r = got.detach().double().cpu(), ref.detach().double().cpu()
    return ((g - r).abs().max() / r.abs().max().clamp_min(1e-30)).item()


def call(name, *args):
    from vit_grid_model_b200 import _lib
    from vit_grid_model_b200.ops import _st
    _lib.call(name, *args, _st())


def p_(t):
    return None if t is None else t.data_ptr()


# =========================================================================================== 1. kernels, three "ranks"
SPLITS = (500, 300, 150)           # 500: not a multiple of 256; 150: below 256.  Multiples of the 50-row fields of fgate / fadd
HW = 50


def _stats_split(X, gamma, beta, rm, rv, eps=1e-5, mom=0.1):
    C = X.shape[1]
    from vit_grid_model_b200 import _lib
    rows, lo = [], 0
    for Mr in SPLITS:
        row = torch.full((2 * C + 1,), float("nan"), dtype=F64, device=DEV)
        work = torch.empty(max(1, _lib.load().vg_bn_workspace(Mr, C)), device=DEV)
        call("vg_bn_stats_local", X[lo:lo + Mr].data_ptr(), Mr, C, row.data_ptr(), work.data_ptr(), work.numel())
        rows.append(row)
        lo += Mr
    rows = torch.stack(rows)

    def glob():
        st = torch.full((4, C), float("nan"), device=DEV)
        count = torch.full((1,), float("nan"), dtype=F64, device=DEV)
        rm_, rv_ = rm.clone(), rv.clone()
        call("vg_bn_stats_global", rows.data_ptr(), len(SPLITS), C, gamma.data_ptr(), beta.data_ptr(), eps, mom, rm_.data_ptr(),
             rv_.data_ptr(), st[0].data_ptr(), st[1].data_ptr(), st[2].data_ptr(), st[3].data_ptr(), count.data_ptr())
        return st, count, rm_, rv_
    return rows, glob


@pytest.mark.parametrize("C", [128, 512, 1536, 2048])
def test_bn_stats_split_matches_float64(C):
    """measured on a B200 at 1000 W: mean / rstd / scale / shift / running buffers <= 6.5e-7 of the largest entry at every C
    (rstd at C = 2048 the largest), bound 2.6e-6; the global kernels twice: identical bits"""
    M = sum(SPLITS)
    g = torch.Generator(device=DEV).manual_seed(C)
    X = torch.randn(M, C, generator=g, device=DEV) * 2 + torch.randn(C, generator=g, device=DEV)
    gamma = torch.randn(C, generator=g, device=DEV)
    beta = torch.randn(C, generator=g, device=DEV)
    rm = torch.randn(C, generator=g, device=DEV)
    rv = torch.rand(C, generator=g, device=DEV) + 0.5
    rows, glob = _stats_split(X, gamma, beta, rm, rv)
    st, count, rm1, rv1 = glob()
    st2, count2, rm2, rv2 = glob()
    torch.cuda.synchronize()
    for a, b in ((st, st2), (count, count2), (rm1, rm2), (rv1, rv2)):
        assert torch.equal(a, b)
    assert count.item() == M and [r[2 * C].item() for r in rows] == list(SPLITS)
    X64 = X.double()
    m64 = X64.mean(0)
    var64 = X64.var(0, unbiased=False)
    r64 = (var64 + 1e-5).rsqrt()
    sc64 = gamma.double() * r64
    ref = dict(mean=m64, rstd=r64, scale=sc64, shift=beta.double() - m64 * sc64,
               run_mean=0.9 * rm.double() + 0.1 * m64, run_var=0.9 * rv.double() + 0.1 * X64.var(0, unbiased=True))
    got = dict(mean=st[0], rstd=st[1], scale=st[2], shift=st[3], run_mean=rm1, run_var=rv1)
    errs = {k: rel(got[k], ref[k]) for k in ref}
    note(C=C, **errs)
    assert max(errs.values()) < 2.6e-6, errs


@pytest.mark.parametrize("se", [False, True], ids=["plain", "fgate_fadd"])
@pytest.mark.parametrize("act", [0, 1])
@pytest.mark.parametrize("C", [128, 512, 1536, 2048])
def test_bn_bwd_split_matches_float64(C, act, se):
    """draw of each rank's rows against float64 autograd over the concatenation, and each rank's local dgamma / dbeta against
    float64 sums of its rows.  measured on a B200 at 1000 W: draw <= 2.9e-7, dgamma / dbeta <= 9.4e-7 of the largest entry
    (dbeta at C = 1536, GELU, fgate / fadd the largest), bound 3.8e-6; the global kernel twice: identical bits"""
    from vit_grid_model_b200 import _lib
    M = sum(SPLITS)
    g = torch.Generator(device=DEV).manual_seed(7 * C + act)
    X = torch.randn(M, C, generator=g, device=DEV) * 2 + 0.5
    gamma = torch.randn(C, generator=g, device=DEV)
    beta = torch.randn(C, generator=g, device=DEV)
    dOut = torch.randn(M, C, generator=g, device=DEV)
    fgate = torch.rand(M // HW, C, generator=g, device=DEV) if se else None
    fadd = torch.randn(M // HW, C, generator=g, device=DEV) * 0.1 if se else None
    rm, rv = torch.zeros(C, device=DEV), torch.ones(C, device=DEV)
    _, glob = _stats_split(X, gamma, beta, rm, rv)
    st, count, _, _ = glob()
    # float64 reference: autograd over the concatenated rows, the upstream gradient g = dOut*fgate[n] + fadd[n]
    X64 = X.double().requires_grad_(True)
    y = F.batch_norm(X64[:, :, None], None, None, gamma.double(), beta.double(), True, 0.0, 1e-5)[:, :, 0]
    a = F.gelu(y) if act == 1 else y
    up = dOut.double()
    if se:
        up = up * fgate.double().repeat_interleave(HW, 0) + fadd.double().repeat_interleave(HW, 0)
    (a * up).sum().backward()
    draw_ref = X64.grad
    with torch.no_grad():
        xhat = (X64 - X64.mean(0)) * (X64.var(0, unbiased=False) + 1e-5).rsqrt()
        dpre = up * _act_grad(xhat * gamma.double() + beta.double(), act)
    rows, lo, local = [], 0, []
    for r, Mr in enumerate(SPLITS):
        dg0 = torch.randn(C, generator=g, device=DEV) * 0.01
        db0 = torch.randn(C, generator=g, device=DEV) * 0.01
        dg, db = dg0.clone(), db0.clone()
        row = torch.full((2 * C,), float("nan"), dtype=F64, device=DEV)
        work = torch.empty(max(1, _lib.load().vg_bn_workspace(Mr, C)), device=DEV)
        fg = fgate[lo // HW:(lo + Mr) // HW] if se else None
        fa = fadd[lo // HW:(lo + Mr) // HW] if se else None
        call("vg_bn_bwd_local", dOut[lo:lo + Mr].data_ptr(), X[lo:lo + Mr].data_ptr(), st[2].data_ptr(), st[3].data_ptr(),
             st[0].data_ptr(), st[1].data_ptr(), act, p_(fg), p_(fa), HW if se else 0, Mr, C, dg.data_ptr(), db.data_ptr(),
             row.data_ptr(), work.data_ptr(), work.numel())
        rows.append(row)
        local.append((dg - dg0, db - db0, (dpre[lo:lo + Mr] * xhat[lo:lo + Mr]).sum(0), dpre[lo:lo + Mr].sum(0), fg, fa))
        lo += Mr
    rows = torch.stack(rows)
    errs = {}
    for rep in range(2):
        lo, draws = 0, []
        for r, Mr in enumerate(SPLITS):
            draw = torch.full((Mr, C), float("nan"), device=DEV)
            work = torch.empty(2 * C, device=DEV)
            fg, fa = local[r][4], local[r][5]
            call("vg_bn_bwd_global", dOut[lo:lo + Mr].data_ptr(), X[lo:lo + Mr].data_ptr(), st[2].data_ptr(), st[3].data_ptr(),
                 st[0].data_ptr(), st[1].data_ptr(), gamma.data_ptr(), act, p_(fg), p_(fa), HW if se else 0, Mr, C,
                 rows.data_ptr(), len(SPLITS), count.data_ptr(), draw.data_ptr(), work.data_ptr(), work.numel())
            draws.append(draw)
            lo += Mr
        draw = torch.cat(draws)
        if rep == 0:
            first = draw
        else:
            torch.cuda.synchronize()
            assert torch.equal(first, draw)
    errs["draw"] = max(rel(draw[lo:lo + Mr], draw_ref[lo:lo + Mr]) for lo, Mr in zip((0, 500, 800), SPLITS))
    errs["dgamma"] = max(rel(dg, ref_dg) for dg, _, ref_dg, _, _, _ in local)
    errs["dbeta"] = max(rel(db, ref_db) for _, db, _, ref_db, _, _ in local)
    note(C=C, act=act, se=se, **errs)
    assert max(errs.values()) < 3.8e-6, errs


def _act_grad(u, act):
    if act == 0:
        return torch.ones_like(u)
    return 0.5 * (1 + torch.erf(u / 2 ** 0.5)) + u * torch.exp(-0.5 * u * u) / (2 * torch.pi) ** 0.5


# =========================================================================================== 2-5. spawned ranks
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _spawn(case, world, backend, **kw):
    """run _case_<case>(rank, world, **kw) in `world` spawned processes -> [result of rank 0, result of rank 1, ...]"""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, backend, case, kw, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = {}
    try:
        for _ in range(world):
            rank, blob = q.get(timeout=900)
            res[rank] = torch.load(io.BytesIO(blob), weights_only=False)
    finally:
        for p in procs:
            p.join(timeout=120)
    for p in procs:
        assert p.exitcode == 0, p.exitcode
    for r in range(world):
        if isinstance(res[r], BaseException):
            raise res[r]
    return [res[r] for r in range(world)]


def _worker(rank, world, port, backend, case, kw, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    try:
        torch.cuda.set_device(rank if backend == "nccl" else 0)
        if backend is not None:                      # None: the case initialises (or not) torch.distributed itself
            dist.init_process_group(backend, rank=rank, world_size=world)
        out = globals()["_case_" + case](rank, world, **kw)
    except BaseException as e:                       # re-raised by the parent
        import traceback
        out = RuntimeError(f"rank {rank}: {traceback.format_exc()}")
    finally:
        if dist.is_initialized():
            dist.destroy_process_group()
    buf = io.BytesIO()                                # bytes, not shared-memory tensors: the process exits after the put
    torch.save(out, buf)
    q.put((rank, buf.getvalue()))


def _metnet3(cfg, precision, convert, seed=0):
    from vit_grid_model_b200 import MetNet3
    m = MetNet3(**cfg.metnet3_kwargs(), dropout=0.0)
    m.load_state_dict(synth.make_state_dict(synth.metnet3_spec(cfg), seed=seed), strict=True)
    if convert:
        m = nn.SyncBatchNorm.convert_sync_batchnorm(m)
    return m.cuda().train().set_precision(precision)


MV = dict(dim=512, heads=32, dim_head=64, window=8, R=4, N=4, H=16)


def _maxvit(precision, convert):
    from vit_grid_model_b200 import MaxViT
    m = MaxViT(dim=MV["dim"], depth=1, cond_dim=2, heads=MV["heads"], dim_head=MV["dim_head"], vit_window_size=MV["window"],
               num_register_tokens=MV["R"], dropout=0.0)
    m.load_state_dict(synth.make_state_dict(_maxvit_spec(), seed=2), strict=True)
    if convert:
        m = nn.SyncBatchNorm.convert_sync_batchnorm(m)
    return m.cuda().train().set_precision(precision)


def _maxvit_spec():
    return synth.maxvit_spec(MV["dim"], 1, 2, MV["heads"], MV["dim_head"], MV["window"], 4, 0.25, MV["R"])


def _maxvit_inputs():
    g = torch.Generator().manual_seed(21)
    N, D, H = MV["N"], MV["dim"], MV["H"]
    return torch.randn(N, D, H, H, generator=g), torch.randn(N, 2, generator=g), torch.randn(N, D, H, H, generator=g)


def _avg_grads(m, world):
    """the data-parallel average of p.grad (what GradSync's AVG all-reduce does; gloo has no AVG): one flat SUM all-reduce / world"""
    import torch.distributed as dist
    ps = [p for p in m.parameters()]
    flat = torch.cat([p.grad.reshape(-1) for p in ps])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM)
    flat /= world
    out, off = {}, 0
    for (k, p) in m.named_parameters():
        out[k] = flat[off:off + p.numel()].view(p.shape).cpu()
        off += p.numel()
    return out


def _step(model_kind, precision, convert, B, rank, world, deterministic=False):
    """one data-parallel step on this rank's shard -> dict of CPU tensors (prediction, loss, averaged gradients, buffers)"""
    from vit_grid_model_b200 import focal_r_loss
    from vit_grid_model_b200.parallel import shard_batch
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(deterministic)
    try:
        lo, hi = shard_batch(B, rank, world)
        if model_kind == "metnet3":
            cfg = synth.CFG_SMALL128
            m = _metnet3(cfg, precision, convert)
            x, ts, target = synth.make_inputs(cfg, B, seed=77)
            pred = m(x[lo:hi].cuda(), timestamps=ts[lo:hi].cuda())
            loss = focal_r_loss(pred, target[lo:hi].cuda())
        else:
            m = _maxvit(precision, convert)
            x, cond, w = _maxvit_inputs()
            pred = m(x[lo:hi].cuda(), cond[lo:hi].cuda())
            loss = (pred * w[lo:hi].cuda()).sum() / (hi - lo)
        loss.backward()
        grads = _avg_grads(m, world)
        torch.cuda.synchronize()
        return dict(pred=pred.detach().cpu(), loss=loss.detach().cpu(), grads=grads,
                    buffers={k: b.detach().cpu() for k, b in m.named_buffers()}, span=(lo, hi))
    finally:
        torch.use_deterministic_algorithms(prev)


def _case_step(rank, world, model_kind, precision, B, convert=True, repeat=False):
    out = _step(model_kind, precision, convert, B, rank, world)
    if repeat:
        a = _step(model_kind, precision, convert, B, rank, world, deterministic=True)
        b = _step(model_kind, precision, convert, B, rank, world, deterministic=True)
        out["det_identical"] = _identical(a, b)
    return out


def _identical(a, b):
    flat = lambda d: {f"{k}.{j}": v for k, sub in d.items() if isinstance(sub, dict) for j, v in sub.items()} | \
        {k: v for k, v in d.items() if torch.is_tensor(v)}
    fa, fb = flat(a), flat(b)
    return fa.keys() == fb.keys() and all(torch.equal(fa[k], fb[k]) for k in fa)


# ---- float64 oracle on the whole batch, train mode, running-buffer updates recorded
class _RecordBN:
    """F.batch_norm wrapper: the oracle's train-mode BatchNorm calls (in module order) -> batch mean and unbiased variance"""

    def __init__(self):
        self.stats, self.orig = [], F.batch_norm

    def __enter__(self):
        def bn(x, rm, rv, w=None, b=None, training=False, momentum=0.1, eps=1e-5):
            if training:
                d = x.detach()
                self.stats.append((d.mean((0, 2, 3)), d.var((0, 2, 3), unbiased=True)))
            return self.orig(x, rm, rv, w, b, training, momentum, eps)
        F.batch_norm = bn
        return self

    def __exit__(self, *a):
        F.batch_norm = self.orig


class _PerRankInputs:
    """The reference's time-embedding scramble (quirk Q1, oracle/metnet3_oracle.py:prepare_input) couples every field to the
    timestamps of the other samples of the same forward call, so a rank's fields see its own shard's timestamps: the oracle's
    whole batch is each shard's prepared input, concatenated in rank order (everything after it is per field, BatchNorm aside)"""

    def __init__(self, spans):
        import oracle.metnet3_oracle as mo3
        self.mod, self.spans, self.orig = mo3, spans, mo3.prepare_input

    def __enter__(self):
        def prepare(x, timestamps, sd, cfg, stn_imgs=False, samples=None):
            assert samples is None
            parts = [self.orig(x[lo:hi], timestamps[lo:hi], sd, cfg, stn_imgs) for lo, hi in self.spans]
            return torch.cat([h for h, _ in parts]), torch.cat([c for _, c in parts])
        self.mod.prepare_input = prepare

    def __exit__(self, *a):
        self.mod.prepare_input = self.orig


def _oracle(model_kind, B, spans):
    """-> (pred, per-rank losses, gradients of the mean over ranks of each rank's loss, expected running buffers) in float64"""
    from oracle.focal_r_oracle import focal_r
    from oracle.metnet3_oracle import metnet3_forward
    from oracle import maxvit_oracle as mo
    if model_kind == "metnet3":
        cfg = synth.CFG_SMALL128
        sd = synth.make_state_dict(synth.metnet3_spec(cfg), seed=0)
        x, ts, target = synth.make_inputs(cfg, B, seed=77)
    else:
        sd = synth.make_state_dict(_maxvit_spec(), seed=2)
        x, cond, w = _maxvit_inputs()
    for k, v in sd.items():
        sd[k] = v.to(DEV, F64) if v.is_floating_point() else v.to(DEV)
        if v.is_floating_point() and "running_" not in k and k != "pm25_boundaries":
            sd[k].requires_grad_(True)
    with _RecordBN() as rec:
        if model_kind == "metnet3":
            with _PerRankInputs(spans):
                pred = metnet3_forward(x.to(DEV, F64), ts.cpu(), sd, cfg, training=True)
            losses = [focal_r(pred[lo:hi], target[lo:hi].to(DEV, F64)) for lo, hi in spans]
        else:
            pred = mo.maxvit_forward(x.to(DEV, F64), cond.to(DEV, F64), sd, depth=1, heads=MV["heads"], window=MV["window"],
                                     num_reg=MV["R"], training=True)
            losses = [(pred[lo:hi] * w[lo:hi].to(DEV, F64)).sum() / (hi - lo) for lo, hi in spans]
    (sum(losses) / len(losses)).backward()
    names = sorted({k.rsplit(".", 1)[0] for k in sd if k.endswith(".running_mean")}, key=lambda n: list(sd).index(n + ".running_mean"))
    assert len(names) == len(rec.stats)
    bufs = {}
    for n, (mean, var) in zip(names, rec.stats):
        bufs[n + ".running_mean"] = (0.9 * sd[n + ".running_mean"] + 0.1 * mean).cpu()
        bufs[n + ".running_var"] = (0.9 * sd[n + ".running_var"] + 0.1 * var).cpu()
    grads = {k: v.grad.cpu() for k, v in sd.items() if torch.is_tensor(v) and v.requires_grad}
    return pred.detach().cpu(), [l.item() for l in losses], grads, bufs


def _grad_errors(grads, ref):
    """-> ({name: max error / largest reference entry}, global relative L2).  The biases of the 1x1 / depthwise convolutions in
    front of a batch-statistic BatchNorm have an analytically zero gradient (float64: ~1e-15 of the largest entry); theirs is
    taken relative to the largest entry of all gradients"""
    emaxs, num, den = {}, 0.0, 0.0
    top = max(r.abs().max().item() for r in ref.values())
    for k, g in grads.items():
        r = ref[k]
        rmax = r.abs().max().item()
        emaxs[k] = ((g.double() - r).abs().max() / (top if rmax < 1e-9 * top else max(rmax, 1e-2))).item()
        num += (g.double() - r).pow(2).sum().item()
        den += r.pow(2).sum().item()
    return emaxs, (num / den) ** 0.5


def _cosines(grads, ref):
    bad = []
    for k, g in grads.items():
        r = ref[k]
        if r.norm().item() > 1e-2:
            cos = (torch.dot(g.double().reshape(-1), r.reshape(-1)) / (g.double().norm() * r.norm()).clamp_min(1e-12)).item()
            if cos < 0.95:
                bad.append((k, round(cos, 4)))
    return bad


def _check_against_oracle(res, model_kind, precision, B, label):
    spans = [r["span"] for r in res]
    pred_o, losses_o, grads_o, bufs_o = _oracle(model_kind, B, spans)
    fp32 = precision == "fp32"
    ptol, ltol = (1e-4, 1e-4) if fp32 else (3e-2, 1e-2)          # test_train_gpu.py's rules
    perr = max(rel(r["pred"], pred_o[lo:hi]) for r, (lo, hi) in zip(res, spans))
    lerr = max(abs(r["loss"].item() - lo_) / abs(lo_) for r, lo_ in zip(res, losses_o))
    emaxs, glob = _grad_errors(res[0]["grads"], grads_o)
    berr = max(((res[0]["buffers"][k].double() - v).abs().max() / v.abs().max().clamp_min(1e-3)).item() for k, v in bufs_o.items())
    note(case=label, pred=perr, loss=lerr, grad_max=max(emaxs.values()), grad_l2=glob, buffers=berr)
    assert perr < ptol and lerr < ltol, (perr, lerr)
    if fp32:
        bad = {k: e for k, e in emaxs.items() if e > 2e-2}
        assert not bad and glob < 1e-3, (bad, glob)
        assert berr < 1e-4, berr
    else:
        assert not _cosines(res[0]["grads"], grads_o) and glob < 0.2, (_cosines(res[0]["grads"], grads_o), glob)
        assert berr < 2e-2, berr
    for r in res[1:]:                                 # every rank holds the same averaged gradients and running buffers
        assert all(torch.equal(r["grads"][k], res[0]["grads"][k]) for k in r["grads"])
        assert all(torch.equal(r["buffers"][k], res[0]["buffers"][k]) for k in r["buffers"])
    return glob


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("model_kind", ["metnet3", "maxvit512"])
def test_two_ranks_one_gpu_match_oracle_on_whole_batch(model_kind, precision):
    """gloo, both ranks on cuda:0.  Measured on a B200 at 1000 W -- MetNet3 fp32: prediction 5.3e-6, loss 8e-8, worst gradient
    tensor 3.4e-3, global relative L2 2.8e-4, running buffers 2.1e-6; MetNet3 bf16: prediction 2.3e-2, loss 1.2e-3, global L2
    5.3e-2, buffers 6.4e-4; MaxViT 512 fp32: prediction 5.2e-6, worst tensor 2.8e-5, global L2 1.7e-5, buffers 1.2e-7; MaxViT
    512 bf16: prediction 3.1e-3, loss 6.0e-3, global L2 1.8e-2, buffers 1.2e-4.  Bounds: the fp32 rules of DESIGN.md §2 and the
    mixed-precision rules of test_train_gpu.py.  Two deterministic runs: identical bits"""
    res = _spawn("step", 2, "gloo", model_kind=model_kind, precision=precision, B=4, repeat=True)
    _check_against_oracle(res, model_kind, precision, 4, f"{model_kind}_{precision}_sync")
    assert all(r["det_identical"] for r in res)


@pytest.mark.parametrize("model_kind", ["metnet3", "maxvit512"])
def test_per_rank_statistics_fail_the_whole_batch_check(model_kind):
    """the same two-rank fp32 step without conversion: per-rank statistics move the gradients far outside the global-L2 bound
    the synchronised step meets (measured on a B200: MetNet3 0.27, MaxViT 512 0.67, against the bound 1e-3 that the
    synchronised steps meet at 2.8e-4 and 1.7e-5)"""
    res = _spawn("step", 2, "gloo", model_kind=model_kind, precision="fp32", B=4, convert=False)
    spans = [r["span"] for r in res]
    _, _, grads_o, _ = _oracle(model_kind, 4, spans)
    _, glob = _grad_errors(res[0]["grads"], grads_o)
    note(case=f"{model_kind}_fp32_per_rank", grad_l2=glob)
    assert glob > 1e-3, glob                          # the global-L2 bound of the synchronised fp32 step


def test_unequal_shards_match_oracle():
    """B = 3 over two ranks (2 / 1): predictions, running buffers and the gradients of the mean over ranks of each rank's
    mean loss.  Measured on a B200: prediction 5.6e-6, loss 3.1e-7, worst gradient tensor 2.7e-3, global L2 5.4e-4, running
    buffers 1.7e-6"""
    res = _spawn("step", 2, "gloo", model_kind="metnet3", precision="fp32", B=3)
    assert [r["span"] for r in res] == [(0, 2), (2, 3)]
    _check_against_oracle(res, "metnet3", "fp32", 3, "metnet3_fp32_unequal")


# ---- 4. nothing changes without synchronisation
def _everything(m, x, ts, train):
    from vit_grid_model_b200 import focal_r_loss
    cfg = synth.CFG_SMALL128
    _, _, target = synth.make_inputs(cfg, x.shape[0], seed=77)
    xin = x.clone().requires_grad_(True)
    out = {}
    if train:
        pred = m(xin, timestamps=ts)
        loss = focal_r_loss(pred, target.cuda())
        loss.backward()
        out.update(loss=loss.detach(), pred=pred.detach(), xgrad=xin.grad)
        out.update({"grad." + k: p.grad for k, p in m.named_parameters()})
    else:
        with torch.no_grad():
            out["infer"] = m(x, timestamps=ts)
        pred = m(xin, timestamps=ts)                                    # the frozen eval() x.grad graph
        pred.square().sum().backward()
        out.update(frozen_pred=pred.detach(), xgrad=xin.grad)
    out.update({"buf." + k: b for k, b in m.named_buffers()})
    torch.cuda.synchronize()
    return {k: v.detach().cpu().clone() for k, v in out.items()}


def _case_unsynced(rank, world, precision):
    import torch.distributed as dist
    torch.use_deterministic_algorithms(True)          # bit-comparable steps (the atomic reductions would differ run to run)
    cfg = synth.CFG_SMALL128
    x, ts, _ = synth.make_inputs(cfg, 2, seed=77)
    x, ts = x.cuda(), ts.cuda()
    same = {}
    for train in (True, False):
        mode = "train" if train else "eval"
        ref = _everything(_metnet3(cfg, precision, False).train(train), x, ts, train)
        conv = _everything(_metnet3(cfg, precision, True).train(train), x, ts, train)       # torch.distributed not initialised
        same[f"{mode}_no_process_group"] = _identical(ref, conv)
        dist.init_process_group("gloo", rank=0, world_size=1)
        try:
            conv1 = _everything(_metnet3(cfg, precision, True).train(train), x, ts, train)  # a one-rank WORLD
            same[f"{mode}_one_rank_group"] = _identical(ref, conv1)
        finally:
            dist.destroy_process_group()
    return same


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_without_sync_the_converted_model_gives_the_same_bits(precision):
    res = _spawn("unsynced", 1, None, precision=precision)[0]
    assert all(res.values()), res


# ---- 5. two GPUs over NCCL
def _case_nccl(rank, world):
    import torch.distributed as dist
    from vit_grid_model_b200 import DataParallel, FlatAdamW, focal_r_loss
    from vit_grid_model_b200.parallel import shard_batch
    cfg = synth.CFG_SMALL128
    B = 4
    m = _metnet3(cfg, "fp32", True)
    ddp = DataParallel(m)
    assert ddp.stats_group is not None
    opt = FlatAdamW(m, lr=1e-4, weight_decay=0.01)
    lo, hi = shard_batch(B, rank, world)
    x, ts, target = synth.make_inputs(cfg, B, seed=77)
    pred = ddp(x[lo:hi].cuda(), timestamps=ts[lo:hi].cuda())
    loss = focal_r_loss(pred, target[lo:hi].cuda())
    loss.backward()
    grads = {k: p.grad.detach().cpu().clone() for k, p in m.named_parameters()}       # already averaged by GradSync
    buffers = {k: b.detach().cpu().clone() for k, b in m.named_buffers()}
    opt.step()
    torch.cuda.synchronize()
    after = {k: t.detach().cpu().clone() for k, t in list(m.named_parameters()) + list(m.named_buffers())}
    return dict(pred=pred.detach().cpu(), loss=loss.detach().cpu(), grads=grads, buffers=buffers, after=after, span=(lo, hi))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_gpus_nccl_data_parallel_matches_oracle():
    """the bounds of the gloo fp32 case (not yet measured: it has not run on a two-GPU host); parameters and
    buffers after one FlatAdamW step: identical bits on both ranks"""
    res = _spawn("nccl", 2, "nccl")
    _check_against_oracle(res, "metnet3", "fp32", 4, "metnet3_fp32_nccl")
    assert all(torch.equal(res[1]["after"][k], v) for k, v in res[0]["after"].items())
