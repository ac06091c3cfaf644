"""Shared helpers for the parity tests."""
import glob
import os

import torch

from graphgps_b200.batch import GraphBatch

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden_names():
    return sorted(os.path.basename(p)[:-3] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.pt")))


def load_golden(name):
    return torch.load(os.path.join(GOLDEN_DIR, name + ".pt"), weights_only=False)


def golden_batch(fix, device="cpu", dtype=torch.float32):
    return GraphBatch(x=fix["x"].to(device=device, dtype=dtype), edge_index=fix["edge_index"].to(device),
                      edge_attr=fix["edge_attr"].to(device=device, dtype=dtype), batch=fix["batch"].to(device),
                      num_graphs=fix["num_graphs"])


def run_layer(layer, batch, fix, backward=True):
    """forward (+backward with the fixture's cotangents). Returns dict of outputs/grads on CPU."""
    cfg = fix["config"]
    batch.x.requires_grad_(backward)
    batch.edge_attr.requires_grad_(backward)
    x_in, e_in = batch.x, batch.edge_attr
    out = layer(batch)
    res = {"out_x": out.x.detach().cpu()}
    dev, dt = out.x.device, out.x.dtype
    loss = (out.x * fix["ct_x"].to(device=dev, dtype=dt)).sum()
    if cfg["local"] == "CustomGatedGCN":
        res["out_e"] = out.edge_attr.detach().cpu()
        loss = loss + (out.edge_attr * fix["ct_e"].to(device=dev, dtype=dt)).sum()
    if backward:
        loss.backward()
        res["grad_x"] = x_in.grad.detach().cpu()
        if e_in.grad is not None:
            res["grad_e"] = e_in.grad.detach().cpu()
        res["grad_params"] = {n: p.grad.detach().cpu() for n, p in layer.named_parameters() if p.grad is not None}
    res["state_after"] = {k: v.detach().cpu() for k, v in layer.state_dict().items()
                          if "running" in k or "num_batches" in k}
    return res


def load_reference_golden(name):
    """tests/golden/reference/<name>.pt: sampled outputs of the reference's own layer files (make_golden.py)."""
    return torch.load(os.path.join(GOLDEN_DIR, "reference", name + ".pt"), weights_only=False)


def sample_summary(tensors, k, seed=0):
    """What a reference golden keeps of each named tensor, in fp64: k entries at fixed, seeded positions (all of a
    smaller tensor) and the full tensor's sum, sum of magnitudes and largest magnitude."""
    g = torch.Generator().manual_seed(seed)
    names, count, numel, idx, val, stats = [], [], [], [], [], []
    for n, t in tensors.items():
        f = t.detach().cpu().double().flatten()
        i = torch.randperm(f.numel(), generator=g)[:k]
        names.append(n)
        count.append(i.numel())
        numel.append(f.numel())
        idx.append(i.int())
        val.append(f[i])
        stats.append(torch.stack([f.sum(), f.abs().sum(), f.abs().max()]))
    return {"names": names, "count": count, "numel": numel, "idx": torch.cat(idx), "val": torch.cat(val),
            "stats": torch.stack(stats)}


def check_summary(tensors, summ, tol, what, scaled=False):
    """Asserts what max|a - b| <= tol * s implies for every tensor of a sample_summary: each stored entry within
    tol * s, the sum, the sum of magnitudes within numel * tol * s, and the largest magnitude within tol * s.
    s = 1, or max(1, max|b|) when scaled."""
    assert sorted(tensors) == sorted(summ["names"]), (what, sorted(set(tensors) ^ set(summ["names"])))
    bad, off = {}, 0
    for n, c, ne, st in zip(summ["names"], summ["count"], summ["numel"], summ["stats"]):
        f = tensors[n].detach().cpu().double().flatten()
        i, v = summ["idx"][off:off + c].long(), summ["val"][off:off + c]
        off += c
        if f.numel() != ne:
            bad[n] = ("numel", f.numel(), ne)
            continue
        s = max(1.0, float(st[2])) if scaled else 1.0
        got = torch.stack([f.sum(), f.abs().sum(), f.abs().max()])
        err = max(float((f[i] - v).abs().max()) / s, float((got[:2] - st[:2]).abs().max()) / (ne * s),
                  float((got[2] - st[2]).abs()) / s)
        if not err <= tol:
            bad[n] = err
    assert not bad, f"{what}: tolerance {tol} exceeded: {bad}"


def rel_err(a, b):
    """max |a-b| / max(1, max|b|): absolute on O(1) (BatchNorm-normalised) data, relative on large."""
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / max(1.0, float(b.abs().max())))


def rel_l2(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / max(float(b.norm()), 1e-30))


def compare(res, fix, tol, what="", grad_l2_tol=None):
    """Forward outputs and BatchNorm running statistics: max|a-b| / max(1, max|b|) <= tol.

    Gradients: the same max-abs criterion, OR (when grad_l2_tol is given) relative L2 error
    <= grad_l2_tol.  The second criterion exists because the derivative of a ReLU network is
    discontinuous: a pre-activation within rounding distance of 0 flips its mask between two
    correct arithmetics (the reference's own fp32 vs fp64 runs differ by 1.8e-2 max-abs on
    ff_linear1.weight at the code2 shape for exactly this reason), which moves a handful of
    gradient entries by O(|g|) while leaving the L2 error at the rounding level.  A real defect
    (wrong operand, missing term) shows up as an L2 error of order 1.
    """
    errs, bad = {}, {}

    def check_fwd(key, a, b):
        e = rel_err(a, b)
        errs[key] = e
        errs["raw:" + key] = float((a.double() - b.double()).abs().max())   # unscaled max-abs beside the scaled one
        if not e <= tol:
            bad[key] = e

    def check_grad(key, a, b):
        e = rel_err(a, b)
        errs[key] = e
        errs["raw:" + key] = float((a.double() - b.double()).abs().max())
        if e <= tol:
            return
        if grad_l2_tol is not None:
            l2 = rel_l2(a, b)
            errs[key + "(l2)"] = l2
            if l2 <= grad_l2_tol:
                return
            bad[key] = (e, l2)
        else:
            bad[key] = e

    for k in ("out_x", "out_e"):
        if k in fix and k in res:
            check_fwd(k, res[k], fix[k])
    for k in ("grad_x", "grad_e"):
        if k in fix and k in res:
            check_grad(k, res[k], fix[k])
    for n, g in fix.get("grad_params", {}).items():
        if n in res.get("grad_params", {}):
            check_grad("grad:" + n, res["grad_params"][n], g)
        else:
            bad["grad:" + n] = float("inf")
    for n, v in fix.get("state_after", {}).items():
        if v.is_floating_point():
            check_fwd("state:" + n, res["state_after"][n], v)
        elif bool((res["state_after"][n] != v).any()):
            bad["state:" + n] = 1.0
    assert not bad, f"{what} tolerance {tol} (grad L2 {grad_l2_tol}) exceeded: {bad}"
    return errs
