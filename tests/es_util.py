"""Helpers of the EquivStableLapPE tests: the fixtures under tests/golden/eslappe/ (make_golden.py ES_CASES) and a
run_layer that also feeds batch.pe_EquivStableLapPE and returns its gradient."""
import glob
import os

import torch

from util import GOLDEN_DIR, golden_batch, rel_l2, run_layer

ES_DIR = os.path.join(GOLDEN_DIR, "eslappe")


def es_golden_names():
    return sorted(os.path.basename(p)[:-3] for p in glob.glob(os.path.join(ES_DIR, "*.pt")))


def load_es_golden(name):
    return torch.load(os.path.join(ES_DIR, name + ".pt"), weights_only=False)


def es_batch(fix, device="cpu", dtype=torch.float32, pe_grad=True):
    b = golden_batch(fix, device, dtype)
    b.pe_EquivStableLapPE = fix["pe"].to(device=device, dtype=dtype).requires_grad_(pe_grad)
    return b


def run_es_layer(layer, batch, fix, backward=True):
    """util.run_layer plus res["grad_pe"] (None when the PE got no gradient)."""
    pe = batch.pe_EquivStableLapPE
    res = run_layer(layer, batch, fix, backward=backward)
    if backward:
        res["grad_pe"] = pe.grad.detach().cpu() if pe.grad is not None else None
    return res


def es_l2_errors(res, fix):
    """Relative L2 errors of the gradients a max-abs bound cannot see: the PE gradient and the mlp_r_ij gradients."""
    out = {"grad_pe": rel_l2(res["grad_pe"], fix["grad_pe"])}
    for n, g in fix["grad_params"].items():
        if "mlp_r_ij" in n:
            out[n] = rel_l2(res["grad_params"][n], g)
    return out
