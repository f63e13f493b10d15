"""Dropout-on training against the fp64 oracle, and the model-level fused operators (include/gnnfd_b200.h section (6)) at
their edges.

The kernels never materialise a dropout mask: they re-derive the keep bits from (seed, position) in the forward and in the
backward.  ``functional.dropout_mask`` exports the same bits, so the oracle can be handed exactly the masks (and the
survivor scale, 65536 / (65536 - floor(p * 65536)), not 1/(1-p)) a training step used:
  * attention: ``[E',8]`` from ``conv.last_dropout_seed``;
  * features:  ``[N*C]`` keyed ``(row_base + n) * C + c`` from the seed ``fused._draw_seed`` hands the BatchNorm tail.

Every comparison prints ``[max-err]`` lines (run with ``-s`` to see the measured maxima next to their bars)."""
import copy
import struct

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from gnn_fraud_detection_b200 import GAT, TemporalGNN, _abi, fused, synth
from gnn_fraud_detection_b200 import functional as Fn
from gnn_fraud_detection_b200.graph import _stream
from oracle import pyg_gatconv as O
from util import maxabs, relerr

pytestmark = pytest.mark.gpu


def _report(name, errs):
    print(f"[max-err] {name}: " + ", ".join(f"{k}={v[0]:.3g} (bar {v[1]:.3g})" for k, v in errs.items()))


def _need_free_bytes(n):
    free_b, _ = torch.cuda.mem_get_info()
    if free_b < n:
        pytest.skip(f"needs {n / 1e9:.0f} GB of free device memory")


def _drel(a, b):
    """relerr on the device (the large cases would spend seconds copying to the host)."""
    a, b = a.detach().double(), b.detach().double()
    return float((a - b).norm() / (b.norm() + 1e-30))


def _dmax(a, b):
    return float((a.detach().double() - b.detach().double()).abs().max()) if a.numel() else 0.0


# ---- B1 / B2: the models with dropout on, against the fp64 oracle given the kernels' masks ---------------------------
class _SeedRecorder:
    """Stands in for ``fused._draw_seed``: the feature-dropout seeds are drawn as before and kept."""

    def __init__(self):
        self.draw, self.seeds = fused._draw_seed, []

    def __call__(self):
        s = self.draw()
        self.seeds.append(s)
        return s


def _data():
    x, ei, _ = synth.elliptic_synth(num_nodes=20_000, num_edges=23_000, num_feats=166, seed=0)
    y = (torch.rand(x.size(0), generator=torch.Generator().manual_seed(1)) < 0.1).long()
    y[::7] = -1
    return x, ei, y


def _pair(cls, p, algo):
    torch.manual_seed(0)
    ref = (O.OracleGAT if cls is GAT else O.OracleTemporalGNN)(166, 64, 1, num_layers=3, dropout=p).double()
    ours = cls(166, 64, 1, num_layers=3, dropout=p, gemm_algo=algo)
    ours.load_state_dict({k: v.float() for k, v in ref.state_dict().items()}, strict=True)
    ref.load_state_dict({k: v.double() for k, v in ours.state_dict().items()}, strict=True)   # identical fp32 values
    return ref.train(), ours.cuda().train()


def _masks(att_seeds, feat_seeds, p, n_edges, N, dev):
    att = [Fn.dropout_mask(s, p, n_edges, 8, dev)[0].cpu() for s in att_seeds]
    feat, scale = [], None
    for s in feat_seeds:
        k, scale = Fn.dropout_mask(s, p, N * 64, 1, dev)
        feat.append(k.view(N, 64).cpu())
    return att, feat, scale


class _LeakyFollow:
    """Stands in for torch.nn.functional inside the oracle module: the attention logits' leaky ReLU takes, layer by layer,
    the branch given in ``branches`` (``[E',H]`` in edge_index' order) -- within 1e-5 of the kink only."""

    def __init__(self, branches):
        self.branches, self.layer, self.forced = branches, 0, 0

    def __getattr__(self, name):
        return getattr(F, name)

    def leaky_relu(self, z, negative_slope):
        want = self.branches[self.layer]
        self.layer += 1
        flip = (z > 0) != want
        if bool(flip.any()):
            far = float(z.detach()[flip].abs().max())
            assert far <= 1e-5, f"the kernel's leaky-ReLU branch differs {far:.3g} away from the kink"
            self.forced += int(flip.sum())
        return z * torch.where(want, torch.ones_like(z), torch.full_like(z, negative_slope))


def _oracle_step(ref, x, ei, y, att, feat, scale, capture_last_bn=False, relu_follow=None, leaky_follow=None):
    """fp64 forward / masked BCE(pos_weight=50) / backward of the oracle with the given masks; (logits, loss, grads, the last
    BatchNorm's output, the number of branches taken from ``relu_follow`` and ``leaky_follow``).

    ``relu_follow``: per layer, the branch the fused BatchNorm tail's ReLU took for every unit (``_relu_decisions``).  Where
    the fp64 pre-activation lies within fp32 reach of the kink (1e-5), fp32 and fp64 may land on different sides of it;
    that unit's gradient then flows in one and not in the other, which alone moves a parameter gradient by up to 1e-3 (one
    such unit in a 20 000-node TemporalGNN step at p = 0.2 did: 43x the gradient bar, 0.1x once the oracle took the
    kernel's branch there).  The oracle takes the kernel's branch at such units (value changed by at most |pre|, gradient
    through as on that side); a disagreement farther from the kink is a failure, not something to follow.
    ``leaky_follow``: the same for the leaky ReLU of the attention logits (``_leaky_decisions``)."""
    ref.zero_grad(set_to_none=True)
    seen = {"forced": 0}
    hooks = []
    if capture_last_bn:
        hooks.append(ref.batch_norms[-1].register_forward_hook(lambda m, i, o: seen.__setitem__("bn", o.detach())))
    if relu_follow is not None:
        def follow(layer):
            def hook(m, inp, o):
                flip = (o > 0) != relu_follow[layer]
                if bool(flip.any()):
                    far = float(o.detach()[flip].abs().max())
                    assert far <= 1e-5, f"layer {layer}: the kernel's ReLU branch differs {far:.3g} away from the kink"
                    seen["forced"] += int(flip.sum())
                return torch.where(flip, o - 2 * o.detach(), o)          # value -o: the other side, gradient 1
            return hook
        hooks += [bn.register_forward_hook(follow(i)) for i, bn in enumerate(ref.batch_norms)]
    kw = {"hidden_state": torch.zeros(x.size(0), 64, dtype=torch.float64)} if isinstance(ref, O.OracleTemporalGNN) else {}
    shim = _LeakyFollow(leaky_follow) if leaky_follow is not None else None
    if shim is not None:
        O.F = shim
    try:
        r = ref(x, ei, att_masks=att, feat_masks=feat, dropout_scale=scale, **kw)
    finally:
        O.F = F
        for h in hooks:
            h.remove()
    if shim is not None:
        seen["forced"] += shim.forced
    lg = r[0] if isinstance(r, tuple) else r
    mask = y != -1
    loss = nn.BCEWithLogitsLoss(pos_weight=torch.tensor(50.0, dtype=torch.float64))(lg[mask].squeeze(1), y[mask].double())
    loss.backward()
    grads = {n: q.grad.detach().clone() for n, q in ref.named_parameters() if "lin_dst" not in n}
    return lg.detach(), float(loss), grads, seen.get("bn"), seen["forced"]


def _record_layer_outputs(model):
    """Keeps the latest output of every GAT layer (the fp32 input of the fused BatchNorm tail).  Under CUDA-graph capture
    the kept tensors are the graph's own buffers, so after a replay they hold that replay's values."""
    outs, ins = [None] * len(model.gat_layers), [None] * len(model.gat_layers)

    def keep(i):
        def hook(m, inp, o):
            ins[i], outs[i] = inp[0], o
        return hook
    for i, conv in enumerate(model.gat_layers):
        conv.register_forward_hook(keep(i))
    return outs, ins


def _relu_decisions(zs, bns):
    """The ReLU branch of every unit as the fused BatchNorm tail takes it, recomputed from the fp32 layer outputs with the
    kernels' arithmetic: fp32 mean and invstd rounded from double column sums (gnnfd_bn_finalize, with float(eps)),
    zhat = (z - mean) * invstd in fp32, and the sign of fmaf(zhat, gamma, beta), which is the sign of the exact
    zhat * gamma + beta and so what double arithmetic gives."""
    out = []
    for z, bn in zip(zs, bns):
        z = z.detach()
        zd = z.double()
        m = zd.sum(0) / z.size(0)
        var = ((zd * zd).sum(0) / z.size(0) - m * m).clamp(min=0)
        eps = float(torch.tensor(bn.eps, dtype=torch.float32))
        zh = (z - m.float()) * (1.0 / torch.sqrt(var + eps)).float()
        pre = zh.double() * bn.weight.detach().double() + bn.bias.detach().double()
        out.append((pre > 0).cpu())
    return out


def _leaky_decisions(model, ins, ei, eg):
    """The leaky-ReLU branch of every attention logit as the kernels take it: the sign of the fp32 a_src[j] + a_dst[i], with
    a_src / a_dst from the layer itself run again on the input it was given (the kernels are deterministic), per edge of
    edge_index' and head."""
    N = ins[0].size(0)
    ei2 = O.rewrite_self_loops(ei, N).to(eg.device)
    out = []
    for conv, h in zip(model.gat_layers, ins):
        g = conv._graph(eg, N)
        xin = h.detach().clone().requires_grad_(h.requires_grad)
        _, a_s, a_d, _, _ = Fn.gatconv(xin, conv.lin_src.weight, conv.att_src, conv.att_dst, conv.bias, g, conv.heads,
                                       conv.out_channels, conv.concat, conv.negative_slope, None, 0.0, conv.feature_dtype,
                                       conv.gemm_algo, want_stats=True)
        out.append(((a_s.detach()[ei2[0]] + a_d.detach()[ei2[1]]) > 0).cpu())
    return out


# Three compounding layers: the bars of tests/test_models_gpu.py -- 2e-4 per gradient, 1e-5 for the logits and the loss.
GRAD_BAR = 2e-4


def _errors(lg, loss, grads, ref_lg, ref_loss, ref_grads):
    """{name: (measured error, bar)}: logits and loss at the bar of tests/test_models_gpu.py, gradients at GRAD_BAR."""
    errs = {}
    if lg is not None:
        errs["logits"] = (relerr(lg, ref_lg), 1e-5)
    errs["loss"] = (abs(loss - ref_loss) / abs(ref_loss), 1e-5)
    assert set(grads) == set(ref_grads)
    for n in ref_grads:
        if n.startswith("gat_layers.") and n.endswith(".bias"):
            # conv biases feed a train-mode BatchNorm: their true gradient is zero, only rounding noise remains
            errs[n] = (maxabs(grads[n], ref_grads[n]), 1e-5)
        else:
            errs[n] = (relerr(grads[n], ref_grads[n]), GRAD_BAR)
    return errs


def _ours_step(m, xg, eg, yg):
    m.zero_grad(set_to_none=True)
    r = m(xg, eg)
    lg = r[0] if isinstance(r, tuple) else r
    loss, _ = fused.masked_bce_with_logits(lg, yg, 50.0)
    loss.backward()
    return lg.detach(), float(loss), {n: q.grad.detach().clone() for n, q in m.named_parameters() if "lin_dst" not in n}


@pytest.mark.parametrize("algo", [_abi.GEMM_AUTO, _abi.GEMM_INPUT], ids=["auto", "input"])
@pytest.mark.parametrize("p", [0.2, 0.5])
@pytest.mark.parametrize("cls", [GAT, TemporalGNN], ids=["GAT", "TemporalGNN"])
def test_dropout_training_matches_the_fp64_oracle_given_the_kernels_masks(cls, p, algo, monkeypatch):
    """Attention dropout and feature dropout together through 3 layers, BatchNorm, residuals, the GRU head and the device
    loss: logits, loss and every parameter gradient against the fp64 oracle fed the masks the step drew."""
    x, ei, y = _data()
    ref, ours = _pair(cls, p, algo)
    rec = _SeedRecorder()
    monkeypatch.setattr(fused, "_draw_seed", rec)
    xg, eg, yg = x.cuda(), ei.cuda(), y.cuda()
    zs, ins = _record_layer_outputs(ours)
    lg, loss, grads = _ours_step(ours, xg, eg, yg)
    follow = _relu_decisions(zs, ours.batch_norms)
    leaky = _leaky_decisions(ours, ins, ei, eg)
    att_seeds = [c.last_dropout_seed for c in ours.gat_layers]
    feat_seeds = list(rec.seeds)
    assert len(feat_seeds) == 3 and None not in att_seeds
    N = x.size(0)
    n_edges = ours.gat_layers[0]._graph(eg, N).n_edges
    att, feat, scale = _masks(att_seeds, feat_seeds, p, n_edges, N, xg.device)
    thr = int(p * 65536)
    assert scale == pytest.approx(65536.0 / (65536 - thr), rel=1e-7)     # the generator's convention, not 1/(1-p)
    ref_lg, ref_loss, ref_grads, bn_last, forced = _oracle_step(ref, x.double(), ei, y, att, feat, scale,
                                                                capture_last_bn=True, relu_follow=follow,
                                                                leaky_follow=leaky)
    errs = _errors(lg, loss, grads, ref_lg, ref_loss, ref_grads)
    _report(f"{cls.__name__} p={p} algo={algo} ({forced} branches at a kink taken from the kernel)", errs)
    for n, (e, bar) in errs.items():
        assert e <= bar, (n, e, bar)

    if p != 0.2:
        return
    # negative controls: the comparison must see a wrong mask.  (a) every mask drawn from seed + 1
    att1, feat1, _ = _masks([s + 1 for s in att_seeds], [s + 1 for s in feat_seeds], p, n_edges, N, xg.device)
    e1 = _errors(lg, loss, grads, *_oracle_step(ref, x.double(), ei, y, att1, feat1, scale)[:3])
    _report(f"{cls.__name__} p={p} algo={algo} NEGATIVE seed+1", e1)
    assert e1["logits"][0] > 10 * e1["logits"][1] and e1["loss"][0] > e1["loss"][1]
    assert sum(e > bar for e, bar in e1.values()) >= len(e1) // 2
    # (b) one feature-mask bit of the last layer flipped: a kept unit with a large positive BatchNorm output at a positive
    # node (pos_weight = 50: the largest per-node gradients)
    w = ref.out.weight.detach()[0].abs()
    score = bn_last.clamp(min=0) * feat[-1].double() * w * (y == 1).double()[:, None]
    n0, c0 = divmod(int(score.argmax()), 64)
    feat2 = [f.clone() for f in feat]
    feat2[-1][n0, c0] = 0
    e2 = _errors(lg, loss, grads, *_oracle_step(ref, x.double(), ei, y, att, feat2, scale, relu_follow=follow,
                                                      leaky_follow=leaky)[:3])
    _report(f"{cls.__name__} p={p} algo={algo} NEGATIVE one feature bit", e2)
    assert e2["logits"][0] > e2["logits"][1]
    assert any(e > bar for n, (e, bar) in e2.items() if n not in ("logits", "loss")), "no gradient sees one wrong mask bit"


@pytest.mark.parametrize("cls", [GAT, TemporalGNN], ids=["GAT", "TemporalGNN"])
def test_graph_replayed_dropout_step_matches_the_fp64_oracle(cls, monkeypatch):
    """DeviceTrainStep replays forward + loss + backward from one CUDA graph and adds a device seed word to every dropout
    seed.  With SGD(lr=0) the weights never move, so ``p.grad`` after a replay is that replay's gradient; the seeds baked
    into the graph are those of the captured (4th) step, and the exported masks add the word's current value."""
    from gnn_fraud_detection_b200.train_step import DeviceTrainStep
    x, ei, y = _data()
    p = 0.2
    ref, ours = _pair(cls, p, _abi.GEMM_AUTO)
    rec = _SeedRecorder()
    monkeypatch.setattr(fused, "_draw_seed", rec)
    xg, eg, yg = x.cuda(), ei.cuda(), y.cuda()
    zs, ins = _record_layer_outputs(ours)
    trainer = None
    try:
        trainer = DeviceTrainStep(ours, xg, eg, yg, optimizer=torch.optim.SGD(ours.parameters(), lr=0.0), pos_weight=50.0,
                                  use_cuda_graph=True)
        assert trainer.graph is not None and len(rec.seeds) == 4 * 3
        att_seeds = [c.last_dropout_seed for c in ours.gat_layers]
        feat_seeds = rec.seeds[-3:]
        N = x.size(0)
        n_edges = ours.gat_layers[0]._graph(eg, N).n_edges
        prev = None
        for replay in range(2):
            loss_d, _ = trainer.step()
            loss = float(loss_d)
            grads = {n: q.grad.detach().clone() for n, q in ours.named_parameters() if "lin_dst" not in n}
            att, feat, scale = _masks(att_seeds, feat_seeds, p, n_edges, N, xg.device)
            if prev is not None:
                assert not torch.equal(prev, att[0])           # each replay draws fresh masks
            prev = att[0]
            follow = _relu_decisions(zs, ours.batch_norms)
            leaky = _leaky_decisions(ours, ins, ei, eg)
            _, ref_loss, ref_grads, _, forced = _oracle_step(ref, x.double(), ei, y, att, feat, scale, relu_follow=follow,
                                                             leaky_follow=leaky)
            errs = _errors(None, loss, grads, None, ref_loss, ref_grads)
            _report(f"{cls.__name__} graph replay {replay + 1} ({forced} branches at a kink taken from the kernel)", errs)
            for n, (e, bar) in errs.items():
                assert e <= bar, (replay, n, e, bar)
    finally:
        if trainer is not None:
            trainer.close()


# ---- B3: the BatchNorm tail ---------------------------------------------------------------------------------------------
def _bn_case(N, C, seed, offset=0.0, affine=True):
    """z [N,C] on the device with no pre-activation within a small band of the ReLU's kink (there an fp32 and an fp64
    evaluation may legitimately disagree on the branch), a BatchNorm with non-trivial parameters and running buffers."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    bn = nn.BatchNorm1d(C, affine=affine).cuda().train()
    with torch.no_grad():
        if affine:
            bn.weight.uniform_(0.5, 1.5, generator=g)
            bn.bias.uniform_(-0.5, 0.5, generator=g)
        bn.running_mean.normal_(generator=g)
        bn.running_var.uniform_(0.5, 2.0, generator=g)
    with torch.no_grad():
        scale = 0.1 if offset else 2.0
        z = (torch.randn(N, C, device="cuda", generator=g) * scale + (offset or 0.5)).double()
        m, sd = z.mean(0), z.var(0, unbiased=False).add(bn.eps).sqrt()
        kink = m - (bn.bias.double() * sd / bn.weight.double() if affine else 0.0)
        band = 1e-3 * sd + 8 * torch.finfo(torch.float32).eps * kink.abs()
        d = z - kink
        z = torch.where(d.abs() < band, kink + torch.where(d >= 0, band, -band), z).float()
    return z, bn


def _bn_reference(z, bn, p, keep, ks, res, d_out):
    """fp64 autograd of bn -> relu -> keep * ks -> + residual, with a copy of ``bn``."""
    rbn = copy.deepcopy(bn).double()
    zr = z.double().requires_grad_(True)
    y = F.relu(rbn(zr))
    if p > 0:
        y = y * keep.double() * ks
    rr = None
    if res is not None:
        rr = res.double().requires_grad_(True)
        y = y + rr
    y.backward(d_out.double())
    return y.detach(), zr.grad, rbn, rr


def _feature_mask(seed, p, N, C):
    if p == 0:
        return None, 1.0
    keep, ks = Fn.dropout_mask(seed, p, N * C, 1, "cuda")
    return keep.view(N, C), ks


def _check_bn(N, C, p, with_res, affine=True, offset=0.0, seed=0):
    z, bn = _bn_case(N, C, seed, offset, affine)
    g = torch.Generator(device="cuda").manual_seed(seed + 1)
    res = torch.randn(N, C, device="cuda", generator=g) if with_res else None
    d_out = torch.randn(N, C, device="cuda", generator=g) / N
    keep, ks = _feature_mask(1234 + seed, p, N, C)
    ref, ref_dz, rbn, _ = _bn_reference(z, bn, p, keep, ks, res, d_out)
    ours = copy.deepcopy(bn)
    zg = z.clone().requires_grad_(True)
    rg = res.clone().requires_grad_(True) if with_res else None
    out = fused.bn_relu_dropout_residual(zg, ours, p, rg, seed=1234 + seed)
    out.backward(d_out)
    # the kernel keeps its batch mean in fp32: its rounding (half an ulp of the mean) shifts every zhat by up to
    # half_ulp * invstd -- the same rounding torch's own fp32 BatchNorm makes.  The bars carry that term.
    mean = z.double().mean(0)
    half_ulp = (torch.nextafter(mean.float().abs(), torch.tensor(float("inf"), device="cuda")) - mean.float().abs()).double() / 2
    invstd = 1.0 / (z.double().var(0, unbiased=False) + bn.eps).sqrt()
    gam = rbn.weight.detach().abs() if affine else torch.ones_like(invstd)
    delta = 1.2 * float((half_ulp * invstd).max())                          # bound on the zhat shift
    shift = delta * float(gam.max()) * ks
    S = float((gam * invstd).max()) * float(d_out.abs().max()) * ks          # magnitude of the terms of dz
    errs = {"out.rel": (_drel(out, ref), 1e-6 + shift), "out.max": (_dmax(out, ref), 1e-5 + shift),
            "dz.max": (_dmax(zg.grad, ref_dz), 1e-5 * S),
            "running_mean": (_drel(ours.running_mean, rbn.running_mean), 1e-6),
            "running_var": (_drel(ours.running_var, rbn.running_var), 1e-6)}
    if N > 2:    # two rows: dz is pure cancellation (its true value is O(eps / var)), only the absolute bar applies
        errs["dz.rel"] = (_drel(zg.grad, ref_dz), 2e-5)
    if affine:
        dbeta = rbn.bias.grad.abs().max()
        errs["dgamma"] = (_dmax(ours.weight.grad, rbn.weight.grad),
                          1e-5 * float(rbn.weight.grad.abs().max()) + float(dbeta) * delta)
        errs["dbeta"] = (_drel(ours.bias.grad, rbn.bias.grad), 1e-5)
    _report(f"bn N={N} C={C} p={p} res={with_res} affine={affine} offset={offset}", errs)
    for n, (e, bar) in errs.items():
        assert e <= bar, (n, e, bar)
    if with_res:
        assert torch.equal(rg.grad, d_out)
    assert int(ours.num_batches_tracked) == int(rbn.num_batches_tracked) == 1
    # the zero pattern (dropped or cut by the ReLU) is exactly the reference's, i.e. the exported mask's
    y, yr = (out.detach() - res, ref - res.double()) if with_res else (out.detach(), ref)
    assert torch.equal(y != 0, yr != 0)


_BN_N = [2, 257, 262_145, 1_000_003]          # 262 145 rows: past the 1024-block cap of the column sums


@pytest.mark.parametrize("with_res", [True, False], ids=["res", "nores"])
@pytest.mark.parametrize("p", [0.0, 0.2, 0.5])
@pytest.mark.parametrize("C", [4, 8, 64, 100, 256])
@pytest.mark.parametrize("N", _BN_N)
def test_bn_tail_with_dropout_against_fp64_autograd(N, C, p, with_res):
    if N * C > 50_000_000:
        _need_free_bytes(40e9)
    _check_bn(N, C, p, with_res, seed=N + C)


@pytest.mark.parametrize("N", [257, 262_145])
def test_bn_tail_without_affine_parameters(N):
    _check_bn(N, 64, 0.2, True, affine=False, seed=7)


def test_bn_tail_large_mean_offset():
    """z = 1e3 + 0.1 randn: the batch variance is computed in one pass, E[z^2] - m^2, in double."""
    _check_bn(262_145, 64, 0.2, True, offset=1e3, seed=11)


def test_bn_tail_row_base_split_equals_one_call():
    """Two halves through the C ABI (sums per half, added; finalize with the total count; apply / backward with row_base)
    against one whole call: the same dropout zero pattern, values within 1e-6 (the sums are added in another order)."""
    L = _abi.lib()
    N, C, p, seed, split = 262_145, 64, 0.2, 4321, 100_003
    z, bn = _bn_case(N, C, 3)
    d_out = torch.randn(N, C, device="cuda", generator=torch.Generator(device="cuda").manual_seed(4)) / N
    gamma, beta = bn.weight.detach(), bn.bias.detach()
    ws = fused._ws(N, z.device)
    st = _stream()
    parts = [(0, split), (split, N)]

    def run(parts):
        sums = torch.zeros(2 * C, dtype=torch.float64, device="cuda")
        for r0, r1 in parts:
            s = torch.empty_like(sums)
            _abi.check(L.gnnfd_bn_sums(z[r0:r1].data_ptr(), r1 - r0, C, s.data_ptr(), ws.data_ptr(), ws.numel(), st))
            sums += s
        mean, invstd = torch.empty(C, device="cuda"), torch.empty(C, device="cuda")
        _abi.check(L.gnnfd_bn_finalize(sums.data_ptr(), float(N), C, float(bn.eps), float(bn.momentum), None, None,
                                       mean.data_ptr(), invstd.data_ptr(), st))
        out = torch.empty_like(z)
        for r0, r1 in parts:
            _abi.check(L.gnnfd_bn_relu_drop_res_fwd(z[r0:r1].data_ptr(), r1 - r0, C, mean.data_ptr(), invstd.data_ptr(),
                                                    gamma.data_ptr(), beta.data_ptr(), p, seed, r0, None,
                                                    out[r0:r1].data_ptr(), st))
        bs = torch.zeros(2 * C, dtype=torch.float64, device="cuda")
        for r0, r1 in parts:
            s = torch.empty_like(bs)
            _abi.check(L.gnnfd_bn_bwd_sums(z[r0:r1].data_ptr(), d_out[r0:r1].data_ptr(), r1 - r0, C, mean.data_ptr(),
                                           invstd.data_ptr(), gamma.data_ptr(), beta.data_ptr(), p, seed, r0, s.data_ptr(),
                                           ws.data_ptr(), ws.numel(), st))
            bs += s
        dz, dg, db = torch.empty_like(z), torch.empty(C, device="cuda"), torch.empty(C, device="cuda")
        for r0, r1 in parts:
            _abi.check(L.gnnfd_bn_bwd_apply(z[r0:r1].data_ptr(), d_out[r0:r1].data_ptr(), r1 - r0, C, mean.data_ptr(),
                                            invstd.data_ptr(), gamma.data_ptr(), beta.data_ptr(), p, seed, r0, bs.data_ptr(),
                                            float(N), dz[r0:r1].data_ptr(), dg.data_ptr(), db.data_ptr(), st))
        return out, dz, dg, db

    halves, whole = run(parts), run([(0, N)])
    keep, _ = _feature_mask(seed, p, N, C)
    assert torch.equal(halves[0] == 0, whole[0] == 0)
    assert torch.equal(halves[1] == 0, whole[1] == 0)
    assert not torch.any((whole[0] != 0) & ~keep.bool())                  # dropped units are zero in both
    errs = {n: (_dmax(a, b) / max(float(b.abs().max()), 1e-30), 1e-6)
            for n, a, b in zip(("out", "dz", "dgamma", "dbeta"), halves, whole)}
    _report("bn row_base split", errs)
    for n, (e, bar) in errs.items():
        assert e <= bar, (n, e, bar)


def test_bn_tail_refuses_a_single_row_like_batchnorm1d():
    bn = nn.BatchNorm1d(64).cuda().train()
    with pytest.raises(ValueError, match="Expected more than 1 value per channel"):
        copy.deepcopy(bn).cpu()(torch.randn(1, 64))
    rm = bn.running_mean.clone()
    with pytest.raises(ValueError, match="Expected more than 1 value per channel"):
        fused.bn_relu_dropout_residual(torch.randn(1, 64, device="cuda"), bn, 0.2)
    assert torch.equal(bn.running_mean, rm) and int(bn.num_batches_tracked) == 0
    fused.bn_relu_dropout_residual(torch.randn(2, 64, device="cuda"), bn, 0.2)          # two rows are a batch


# ---- B4: the GRU head ---------------------------------------------------------------------------------------------------
def _gru_case(N, with_state, sat, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    torch.manual_seed(seed)
    gru, lin = nn.GRUCell(64, 64).cuda(), nn.Linear(64, 1).cuda()
    x = torch.randn(N, 64, device="cuda", generator=g) * sat
    h0 = torch.randn(N, 64, device="cuda", generator=g) * sat if with_state else None
    d_out = torch.randn(N, 1, device="cuda", generator=g) / N
    d_h = torch.randn(N, 64, device="cuda", generator=g) / N
    return gru, lin, x, h0, d_out, d_h


def _gru_reference(gru, lin, x, h0, d_out, d_h):
    rg, rl = copy.deepcopy(gru).double(), copy.deepcopy(lin).double()
    xr = x.double().requires_grad_(True)
    hr = h0.double().requires_grad_(True) if h0 is not None else torch.zeros_like(xr)
    h1 = rg(xr, hr)
    out = rl(h1)
    loss = 0
    if d_out is not None:
        loss = loss + (out * d_out.double()).sum()
    if d_h is not None:
        loss = loss + (h1 * d_h.double()).sum()
    loss.backward()
    return out.detach(), h1.detach(), xr.grad, (hr.grad if h0 is not None else None), rg, rl


def _gru_errors(pairs, sat):
    """Normal inputs: the relative bars of tests/test_fused_gpu.py.  Saturated gates (x, h scaled by 30): many true values
    are ~0 (sigmoid / tanh flat), so the bar is absolute, relative to the tensor's largest entry; it is 5e-5 because the
    fp32 pre-activations then sum terms of up to ~100, and their rounding moves a gate that sits near its centre by ~1e-5
    (the same holds for torch's fp32 GRUCell)."""
    errs = {}
    for n, a, b, bar in pairs:
        if sat == 1:
            errs[n] = (_drel(a, b), bar)
        else:
            errs[n] = (_dmax(a, b) / max(float(b.abs().max()), 1e-30), 5e-5)
    return errs


@pytest.mark.parametrize("sat", [1, 30], ids=["normal", "saturated"])
@pytest.mark.parametrize("with_state", [False, True], ids=["zero_state", "state"])
@pytest.mark.parametrize("N", [1, 31, 32, 33, 9_473, 1_000_000])    # 9 473 > 296 blocks x 32 nodes
def test_gru_head_against_fp64_grucell_and_linear(N, with_state, sat):
    gru, lin, x, h0, d_out, d_h = _gru_case(N, with_state, sat, N + 31 * with_state + sat)
    outr, h1r, dxr, dhr, rg, rl = _gru_reference(gru, lin, x, h0, d_out, d_h)
    gg, gl = copy.deepcopy(gru), copy.deepcopy(lin)
    xg = x.clone().requires_grad_(True)
    hg = h0.clone().requires_grad_(True) if with_state else None
    out, h1 = fused.gru_head(xg, gg, gl, hg)
    ((out * d_out).sum() + (h1 * d_h).sum()).backward()
    pairs = [("out", out, outr, 2e-6), ("h_new", h1, h1r, 2e-6), ("dx", xg.grad, dxr, 1e-5),
             ("dw_ih", gg.weight_ih.grad, rg.weight_ih.grad, 1e-5), ("db_ih", gg.bias_ih.grad, rg.bias_ih.grad, 1e-5),
             ("db_hh", gg.bias_hh.grad, rg.bias_hh.grad, 1e-5), ("dw_out", gl.weight.grad, rl.weight.grad, 1e-5),
             ("db_out", gl.bias.grad, rl.bias.grad, 1e-5)]
    if with_state:
        pairs += [("dh_prev", hg.grad, dhr, 1e-5), ("dw_hh", gg.weight_hh.grad, rg.weight_hh.grad, 1e-5)]
    errs = _gru_errors(pairs, sat)
    _report(f"gru N={N} state={with_state} sat={sat}", errs)
    for n, (e, bar) in errs.items():
        assert e <= bar, (n, e, bar)
    if not with_state:
        assert float(gg.weight_hh.grad.abs().max()) == 0.0        # zero state: no gradient reaches W_hh


@pytest.mark.parametrize("which", ["d_out", "d_hnew"])
@pytest.mark.parametrize("with_state", [False, True], ids=["zero_state", "state"])
def test_gru_head_backward_with_a_null_upstream_gradient(which, with_state):
    """gnnfd_gru_head_bwd takes d_out and d_hnew as optional pointers: NULL is a zero upstream gradient."""
    N = 9_473
    gru, lin, x, h0, d_out, d_h = _gru_case(N, with_state, 1, 5 + with_state)
    if which == "d_out":
        d_out = None
    else:
        d_h = None
    _, _, dxr, dhr, rg, rl = _gru_reference(gru, lin, x, h0, d_out, d_h)
    L = _abi.lib()
    w = [gru.weight_ih, gru.weight_hh, gru.bias_ih, gru.bias_hh, lin.weight.view(-1), lin.bias]
    w = [t.detach().contiguous() for t in w]
    grads = [torch.full_like(t, float("nan")) for t in w]
    dx = torch.empty_like(x)
    dhp = torch.empty_like(x) if with_state else None
    gates = torch.empty(2 * N * 192, device="cuda")
    ws = fused._ws(N, x.device)
    _abi.check(L.gnnfd_gru_head_bwd(x.data_ptr(), _abi.ptr(h0), _abi.ptr(d_out), _abi.ptr(d_h), N,
                                    *[t.data_ptr() for t in w], dx.data_ptr(), _abi.ptr(dhp),
                                    *[t.data_ptr() for t in grads], gates.data_ptr(), ws.data_ptr(), ws.numel(), _stream()))
    pairs = [("dx", dx, dxr, 1e-5), ("dw_ih", grads[0], rg.weight_ih.grad, 1e-5), ("db_ih", grads[2], rg.bias_ih.grad, 1e-5),
             ("db_hh", grads[3], rg.bias_hh.grad, 1e-5)]
    if with_state:
        pairs += [("dh_prev", dhp, dhr, 1e-5), ("dw_hh", grads[1], rg.weight_hh.grad, 1e-5)]
    else:
        assert float(grads[1].abs().max()) == 0.0
    if which == "d_out":
        assert float(grads[4].abs().max()) == 0.0 and float(grads[5].abs().max()) == 0.0    # no gradient through the Linear
    else:
        pairs += [("dw_out", grads[4], rl.weight.grad.view(-1), 1e-5), ("db_out", grads[5], rl.bias.grad, 1e-5)]
    errs = _gru_errors(pairs, 1)
    _report(f"gru NULL {which} state={with_state}", errs)
    for n, (e, bar) in errs.items():
        assert e <= bar, (n, e, bar)


# ---- B5: the device loss ------------------------------------------------------------------------------------------------
def _f2b(v):
    return struct.unpack("<i", struct.pack("<f", v))[0]


def _b2f(b):
    return struct.unpack("<f", struct.pack("<i", b))[0]


def sigmoid_boundary(device):
    """The most negative fp32 logit whose fp32 torch.sigmoid is still >= 0.5 on ``device``, by bisection over the bit
    patterns of -t (sigmoid is monotone, so the predicate flips once)."""
    def ok(b):
        return bool(torch.sigmoid(torch.tensor([-_b2f(b)], dtype=torch.float32, device=device))[0] >= 0.5)
    lo, hi = _f2b(0.0), _f2b(1e-5)
    assert ok(lo) and not ok(hi)
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if ok(mid) else (lo, mid)
    return -_b2f(lo), lo


_SPECIAL = [0.0, 1e-9, -1e-9, 1e-7, -1e-7, 1e-6, -1e-6, 20.0, -20.0, 88.0, -88.0, 100.0, -100.0, 1e4, -1e4]


def _bce_reference(logits, y, pw):
    """fp64 restatement of src/train.py:108-149: mean over labelled nodes of pw*y*softplus(-x) + (1-y)*softplus(x), its
    gradient, and the confusion counts of the fp32 rule torch.sigmoid(logit) >= 0.5 evaluated by torch on the device."""
    x = logits.double().view(-1)
    lab = y != -1
    yf = y.clamp(min=0).double()
    sp = lambda v: v.clamp(min=0) + torch.log1p(torch.exp(-v.abs()))             # noqa: E731
    per = pw * yf * sp(-x) + (1 - yf) * sp(x)
    n = int(lab.sum())
    loss = float(per[lab].sum() / n) if n else 0.0
    g = (torch.sigmoid(x) * (pw * yf + 1 - yf) - pw * yf) / max(n, 1)
    g = torch.where(lab, g, torch.zeros_like(g))
    pred = torch.sigmoid(logits.view(-1)) >= 0.5
    pos = y == 1
    counts = [float(n), float((lab & pred & pos).sum()), float((lab & pred & ~pos & (y == 0)).sum()),
              float((lab & ~pred & (y == 0)).sum()), float((lab & ~pred & pos).sum())]
    return loss, g, counts, n


def _check_bce(logits, y, pw, name):
    loss_ref, g_ref, counts, n = _bce_reference(logits, y, pw)
    lg = logits.clone().requires_grad_(True)
    loss, stats = fused.masked_bce_with_logits(lg, y, pw)
    loss.backward()
    assert stats[1:6].tolist() == counts, (name, stats[1:6].tolist(), counts)
    # a float32 loss cannot carry less than its smallest normal number: the absolute floor only matters for a lone
    # well-classified node with |logit| >= 88, whose true loss is below 2^-126
    err_loss = abs(float(loss) - loss_ref)
    bar_loss = 1e-6 * abs(loss_ref) + 1.2e-38
    # gradient: elementwise against the fp64 formula; absolute part = where the true value is saturated to ~0
    atol = 2e-6 * max(pw, 1.0) / max(n, 1)
    ratio = float(((lg.grad.double().view(-1) - g_ref).abs() / (2e-6 * g_ref.abs() + atol)).max())
    errs = {"loss": (err_loss, bar_loss), "grad/bar": (ratio, 1.0)}
    _report(f"bce {name}", errs)
    assert err_loss <= bar_loss, (name, float(loss), loss_ref)
    assert ratio <= 1.0, name


def test_bce_predicate_matches_torch_sigmoid_at_the_fp32_boundary():
    """The confusion counters use the reference's rule, torch.sigmoid(logit) >= 0.5 in fp32 as torch evaluates it on the
    device: that holds for small negative logits too, down to the boundary found here."""
    t_cuda, b_cuda = sigmoid_boundary("cuda")
    t_cpu, b_cpu = sigmoid_boundary("cpu")
    print(f"[boundary] fp32 sigmoid(x) >= 0.5 holds down to x = {t_cuda!r} on CUDA, {t_cpu!r} on the CPU")
    # every fp32 around the CUDA boundary, one node at a time: TP (label 1) iff the rule says positive
    for k in range(-40, 41):
        v = -_b2f(b_cuda + k)
        x = torch.tensor([[v]], device="cuda")
        _, stats = fused.masked_bce_with_logits(x, torch.ones(1, dtype=torch.int64, device="cuda"), 50.0)
        want = bool(torch.sigmoid(x)[0, 0] >= 0.5)
        assert (float(stats[2]) == 1.0) == want, (v, want)
    # a dense sweep of [-2.5e-7, -1e-7]: every fp32 in it, counted at once
    mags = torch.arange(_f2b(1e-7), _f2b(2.5e-7) + 1, dtype=torch.int32, device="cuda").view(torch.float32)
    x = -mags
    y = torch.ones(x.numel(), dtype=torch.int64, device="cuda")
    _, stats = fused.masked_bce_with_logits(x, y, 1.0)
    assert float(stats[2]) == float((torch.sigmoid(x) >= 0.5).sum())


@pytest.mark.parametrize("pw", [1.0, 50.0])
@pytest.mark.parametrize("labels", ["mixed", "none", "all_positive", "all_labelled"])
@pytest.mark.parametrize("N", [1, 2_097_153, 5_000_000])    # 2 097 153: one row past 1024 blocks x 2048 rows
def test_masked_bce_at_its_edges(N, labels, pw):
    g = torch.Generator(device="cuda").manual_seed(N)
    if N == 1:
        for v in _SPECIAL:
            for yv in ((1,) if labels == "all_positive" else (-1,) if labels == "none" else (0, 1)):
                _check_bce(torch.tensor([[v]], device="cuda"), torch.tensor([yv], device="cuda"), pw, f"N=1 x={v} y={yv} pw={pw}")
        return
    logits = torch.randn(N, 1, device="cuda", generator=g) * 3
    # the special values and every fp32 within 64 ulps of the sigmoid boundary, spread over the array
    t, b = sigmoid_boundary("cuda")
    near = [-_b2f(b + k) for k in range(-64, 65)]
    spec = torch.tensor(_SPECIAL + near, device="cuda")
    idx = torch.randperm(N, device="cuda", generator=g)[: spec.numel() * 50]
    logits.view(-1)[idx] = spec.repeat(50)
    if labels == "mixed":
        y = torch.randint(-1, 2, (N,), device="cuda", generator=g)
    elif labels == "none":
        y = torch.full((N,), -1, dtype=torch.int64, device="cuda")
    elif labels == "all_positive":
        y = torch.ones(N, dtype=torch.int64, device="cuda")
    else:
        y = torch.randint(0, 2, (N,), device="cuda", generator=g)
    _check_bce(logits, y, pw, f"N={N} {labels} pw={pw}")
