"""Helpers shared by the GPU parity tests."""
import numpy as np
import torch

from oracle import pyg_gatconv as O


def seeded_params(K, H, C, concat=False, seed=1, bias_scale=0.1):
    """glorot weights exactly as reset_parameters() draws them, under a fixed seed (plus a non-zero bias so
    that the bias path is exercised)."""
    g = torch.Generator().manual_seed(seed)
    W = O.glorot_(torch.empty(H * C, K), g)
    a_s = O.glorot_(torch.empty(1, H, C), g)
    a_d = O.glorot_(torch.empty(1, H, C), g)
    b = torch.randn(H * C if concat else C, generator=g) * bias_scale
    return W, a_s, a_d, b


def load_ckpt(model, path):
    npz = np.load(path)
    sd = {k: torch.from_numpy(npz[k]) for k in npz.files}
    for k in list(sd):
        if k.endswith("lin_src.weight"):
            sd[k.replace("lin_src", "lin_dst")] = sd[k]
    model.load_state_dict(sd, strict=True)
    return model


def oracle_model_outputs(x, ei, y, golden_dir):
    """The arrays of ``tests/golden/make_reference_goldens.reference_outputs`` computed with the oracle's restated wrappers
    (``OracleGAT`` / ``OracleTemporalGNN``) instead of the reference's classes, fp32 eval outputs included."""
    out = {}
    for name, cls, ck in (("gat", O.OracleGAT, "gat_ckpt.npz"), ("tgn", O.OracleTemporalGNN, "tgn_ckpt.npz")):
        m = load_ckpt(cls(x.size(1), 64, 1, num_layers=3), f"{golden_dir}/{ck}").eval()
        with torch.no_grad():
            r32 = m(x, ei)
            kw = {"hidden_state": torch.zeros(x.size(0), 64, dtype=torch.float64)} if name == "tgn" else {}
            r64 = m.double()(x.double(), ei, **kw)
        if name == "tgn":
            out["tgn_logits_f32"], out["tgn_hidden_f32"], out["tgn_logits_f64"], out["tgn_hidden_f64"] = *r32, *r64
        else:
            out["gat_logits_f32"], out["gat_logits_f64"] = r32, r64
    mask = y != -1
    crit = torch.nn.BCEWithLogitsLoss(pos_weight=torch.tensor(50.0, dtype=torch.float64))
    for name, cls, ck in (("gat", O.OracleGAT, "gat_ckpt.npz"), ("tgn", O.OracleTemporalGNN, "tgn_ckpt.npz")):
        m = load_ckpt(cls(x.size(1), 64, 1, num_layers=3, dropout=0.0), f"{golden_dir}/{ck}").double().train()
        kw = {"hidden_state": torch.zeros(x.size(0), 64, dtype=torch.float64)} if name == "tgn" else {}
        r = m(x.double(), ei, **kw)
        logits = r[0] if name == "tgn" else r
        loss = crit(logits[mask].squeeze(1), y[mask].double())
        loss.backward()
        out[f"train_{name}_loss"], out[f"train_{name}_logits"] = loss, logits
        for pn, p in m.named_parameters():
            if "lin_dst" not in pn:
                out[f"train_{name}_grad.{pn}"] = p.grad
    return {k: v.detach() for k, v in out.items()}


def maxabs(a, b):
    return float((a.detach().double().cpu() - b.detach().double().cpu()).abs().max()) if a.numel() else 0.0


def relerr(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))
