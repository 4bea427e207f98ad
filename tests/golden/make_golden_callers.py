"""Generates tests/golden/reference_callers.npz by EXECUTING the reference's own caller functions — `get_optim` and
`train_batch` of models/train_rels.py, `val_batch` of models/eval_rels.py — against the product surface and inputs of
tests/test_reference_callers.py (train_case / eval_case). The definitions are parsed from the reference tree with `ast`
and run unedited apart from this compat shim (INTEGRATION.md section 3): `x.data[0]` (PyTorch-0.3 indexing of a 0-dim
tensor) -> `float(x)`; the `verbose=` keyword of ReduceLROnPlateau (removed from torch) is dropped.

    python tests/golden/make_golden_callers.py
"""
import ast
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "neural-motifs_b200")):
    sys.path.insert(0, p)
OUT = os.path.dirname(os.path.abspath(__file__))

import make_golden as MG  # noqa: E402
from tests import test_reference_callers as RC  # noqa: E402


class _Shim(ast.NodeTransformer):
    def visit_Subscript(self, node):
        self.generic_visit(node)
        if isinstance(node.value, ast.Attribute) and node.value.attr == "data" and \
                isinstance(node.slice, ast.Constant) and node.slice.value == 0:
            return ast.copy_location(ast.Call(func=ast.Name(id="float", ctx=ast.Load()), args=[node.value.value], keywords=[]), node)
        return node

    def visit_Call(self, node):
        self.generic_visit(node)
        if isinstance(node.func, ast.Name) and node.func.id == "ReduceLROnPlateau":
            node.keywords = [k for k in node.keywords if k.arg != "verbose"]
        return node


def _function(path, name, namespace):
    """exec the (shimmed) definition of top-level function `name` of the reference file into `namespace`."""
    tree = ast.parse(open(path).read())
    node = next(n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == name)
    mod = ast.fix_missing_locations(_Shim().visit(ast.Module(body=[node], type_ignores=[])))
    exec(compile(mod, path, "exec"), namespace)
    return namespace[name]


def main():
    import pandas as pd
    import torch
    from torch import optim
    from torch.nn import functional as F
    from torch.optim.lr_scheduler import ReduceLROnPlateau
    from config import BOX_SCALE, IM_SCALE
    from dataloaders.synthetic import SyntheticBlob
    from lib.evaluation.sg_eval import BasicSceneGraphEvaluator
    from lib.pytorch_misc import clip_grad_norm
    g = {}
    detector, orc, state, conf, nb = RC.train_case()
    ns = dict(detector=detector, conf=conf, optim=optim, ReduceLROnPlateau=ReduceLROnPlateau, F=F, pd=pd,
              clip_grad_norm=clip_grad_norm)
    path = os.path.join(MG.REF, "models", "train_rels.py")
    optimizer, scheduler = _function(path, "get_optim", ns)(conf.lr)
    g["train_lrs"] = np.array([grp["lr"] for grp in optimizer.param_groups])
    ns["optimizer"] = optimizer
    before = {n: p.detach().clone() for n, p in detector.named_parameters()}
    detector.train()
    res = _function(path, "train_batch", ns)(SyntheticBlob(nb, "cpu"), verbose=False)
    for k in res.index:
        g["train_" + k] = np.float64(res[k])
    g["train_moved"] = np.array([n for n, p in detector.named_parameters() if not torch.equal(p, before[n])])
    g["train_params"] = RC.param_samples(detector)

    detector, nb, val, conf = RC.eval_case()
    all_pred_entries = []
    ns = dict(detector=detector, conf=conf, val=val, np=np, BOX_SCALE=BOX_SCALE, IM_SCALE=IM_SCALE,
              all_pred_entries=all_pred_entries)
    evaluator = BasicSceneGraphEvaluator.all_modes()
    with torch.no_grad():
        _function(os.path.join(MG.REF, "models", "eval_rels.py"), "val_batch", ns)(0, SyntheticBlob(nb, "cpu"), evaluator)
    for k, v in all_pred_entries[0].items():
        g["eval_" + k] = v
    rec = evaluator["sgcls"].result_dict["sgcls_recall"]
    g["eval_recall"] = np.array([rec[k][0] for k in (20, 50, 100)])
    np.savez_compressed(os.path.join(OUT, "reference_callers.npz"), **g)
    print("wrote", os.path.join(OUT, "reference_callers.npz"), {k: v.shape for k, v in g.items()})


if __name__ == "__main__":
    main()
