"""The caller code of `models/train_rels.py` (get_optim :57-72, train_batch :118-152) and `models/eval_rels.py` (val_batch
:59-86) against the product's API surface (SURVEY.md section 8b "Model API"):
  * the product's `RelModel` class — `detector[b]` (`__getitem__` + `Blob.scatter` protocol), `detector.train()/eval()`,
    `named_parameters()` with the `roi_fmap*` prefixes, the training `Result` fields and the eval 5-tuple,
  * the product's `lib.pytorch_misc.clip_grad_norm`, `lib.evaluation.sg_eval.BasicSceneGraphEvaluator`, `config` constants,
  * `dataloaders.synthetic.SyntheticBlob` standing in for `dataloaders/blob.py:Blob`.
The caller sequence is restated here in this repository's words and held to tests/golden/reference_callers.npz: what the
reference's OWN function definitions computed when tests/golden/make_golden_callers.py executed them, unedited apart
from a small compat shim, against the same product surface and inputs. Neither needs the reference tree at test time.
The one thing that is NOT the product here is the arithmetic of `forward`: the product has no CPU path (by design).
`forward` is therefore delegated to the oracle restatement operating ON THE PRODUCT'S OWN Parameter objects (the oracle
modules are re-pointed at them), so that the callers' `loss.backward()`, `clip_grad_norm(detector.named_parameters())` and
`optimizer.step()` act on the product model. The same step with the product's kernels is held to the oracle on the GPU
(tests/test_model_gpu.py, and tests/test_callers_gpu.py runs the restated caller sequence end to end there)."""
import os
import sys
import types

import numpy as np
import pytest
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_callers.npz")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))


_BUILT = {}


def _build(mode):
    """Product RelModel (CPU-constructed) whose forward is the oracle's arithmetic on the product's own parameters.
    Built once per module (constructing the three VGG fc stacks and the 1.7 GB synthetic state dominates the run time);
    every caller gets the state reloaded."""
    if mode in _BUILT:
        prod, orc, state = _BUILT[mode]
        prod.load_state_dict(state)
        for p in prod.parameters():
            p.requires_grad = True
            p.grad = None
        return prod, orc, state
    from lib.rel_model import RelModel
    from lib.object_detector import Result
    from oracle import model as OM
    from golden.synthetic_state import synthetic_state, CLASSES, RELS, KW

    class ProductSurface(RelModel):
        def forward(self, x, im_sizes, image_offset, gt_boxes=None, gt_classes=None, gt_rels=None, proposals=None,
                    train_anchor_inds=None, return_fmap=False):
            orc = self.__dict__["_orc"]
            orc.train(self.training)
            out = orc(x, im_sizes, image_offset, gt_boxes, gt_classes, gt_rels)
            if self.training:
                return Result(rm_obj_dists=out.rm_obj_dists, rm_obj_labels=out.rm_obj_labels, rel_dists=out.rel_dists,
                              rel_labels=out.rel_labels, obj_preds=out.obj_preds)
            return out

    prod = ProductSurface(CLASSES, RELS, mode=mode, num_gpus=1, require_overlap_det=True, use_resnet=False,
                          use_proposals=False, pass_in_obj_feats_to_decoder=False, pass_in_obj_feats_to_edge=False,
                          rec_dropout=0.1, **KW)
    orc = OM.RelModel(CLASSES, RELS, mode=mode, **KW)
    sd = orc.state_dict()
    state = synthetic_state([(k, tuple(v.shape), v.dtype) for k, v in sd.items()], seed=3)
    prod.load_state_dict(state)
    # re-point every oracle parameter / buffer at the product's object of the same state-dict name
    for name, p in list(prod.named_parameters()) + list(prod.named_buffers()):
        mod = orc
        parts = name.split(".")
        for part in parts[:-1]:
            mod = getattr(mod, part)
        store = mod._parameters if parts[-1] in mod._parameters else mod._buffers
        assert parts[-1] in store, name
        store[parts[-1]] = p
    prod.__dict__["_orc"] = orc                    # (not registered as a submodule: the state dict stays the product's)
    _BUILT[mode] = (prod, orc, state)
    return prod, orc, state


def _ones_masks(orc, n_obj, n_rel, n_img):
    from model_utils import make_masks
    det, top, ctx = make_masks(n_obj, n_rel, n_img, seed=0)
    ones = lambda d: {k: torch.ones_like(v) for k, v in d.items()}
    orc.detector.masks, orc.masks, orc.context.masks = ones(det), ones(top), ones(ctx)


TRAIN_CONF = dict(adam=False, l2=1e-4, lr=6e-3, clip=5.0, mode="sgcls", num_gpus=1, print_interval=100)
PARAM_SAMPLE = 64


def train_case():
    """The product surface with its detector frozen (train_rels.py:51-52), the run's config and one synthetic batch."""
    from dataloaders.synthetic import make_numpy_batch
    detector, orc, state = _build("sgcls")
    for n, param in detector.detector.named_parameters():
        param.requires_grad = False
    B, boxes = 1, 6
    nb = make_numpy_batch(B, seed=5, boxes_per_img=boxes, rels_per_img=5)
    _ones_masks(orc, B * boxes, B * boxes * (boxes - 1), B)
    orc.detector.rng = np.random.RandomState(7)
    return detector, orc, state, types.SimpleNamespace(**TRAIN_CONF), nb


def eval_case():
    """The product surface in eval mode, one synthetic image and the `val` dataset fields val_batch reads."""
    from config import BOX_SCALE, IM_SCALE
    from dataloaders.synthetic import make_numpy_batch
    detector, orc, _ = _build("sgcls")
    detector.eval()
    nb = make_numpy_batch(1, seed=9, boxes_per_img=7, rels_per_img=6)
    val = types.SimpleNamespace(gt_classes=[nb["gt_classes"][:, 1].copy()],
                                relationships=[nb["gt_rels"][:, 1:].copy()],
                                gt_boxes=[nb["gt_boxes"] * BOX_SCALE / IM_SCALE])
    return detector, nb, val, types.SimpleNamespace(mode="sgcls", num_gpus=1)


def param_samples(model):
    """PARAM_SAMPLE seeded elements of every parameter (all of a smaller one), in named_parameters() order."""
    out = []
    for i, (_, p) in enumerate(model.named_parameters()):
        flat = p.detach().reshape(-1)
        if flat.numel() > PARAM_SAMPLE:
            flat = flat[torch.from_numpy(np.random.RandomState(i).randint(0, flat.numel(), PARAM_SAMPLE))]
        out.append(flat)
    return torch.cat(out).numpy()


def test_train_rels_get_optim_and_train_batch_run_against_the_product():
    import pandas as pd
    from torch.nn import functional as F
    from torch.optim.lr_scheduler import ReduceLROnPlateau
    from lib.pytorch_misc import clip_grad_norm
    from dataloaders.synthetic import SyntheticBlob
    gold = np.load(GOLDEN)
    detector, orc, state, conf, nb = train_case()
    B, boxes = 1, 6
    # get_optim: SGD with momentum and L2, the roi_fmap* fc layers at a tenth of the rate; plateau schedule
    named = [(n, p) for n, p in detector.named_parameters() if p.requires_grad]
    optimizer = torch.optim.SGD([{"params": [p for n, p in named if n.startswith("roi_fmap")], "lr": conf.lr / 10.0},
                                 {"params": [p for n, p in named if not n.startswith("roi_fmap")]}],
                                lr=conf.lr, momentum=0.9, weight_decay=conf.l2)
    scheduler = ReduceLROnPlateau(optimizer, "max", patience=3, factor=0.1, threshold=0.0001, threshold_mode="abs",
                                  cooldown=1)
    assert [g["lr"] for g in optimizer.param_groups] == [conf.lr / 10.0, conf.lr] == gold["train_lrs"].tolist()
    assert len(optimizer.param_groups[0]["params"]) == 8              # fc6 / fc7 weights + biases of roi_fmap and roi_fmap_obj
    before = {n: p.detach().clone() for n, p in detector.named_parameters()}
    detector.train()
    # train_batch: detector[b]; object + relation cross-entropies; backward; global-norm clip; step; losses as a Series
    result = detector[SyntheticBlob(nb, "cpu")]
    losses = {"class_loss": F.cross_entropy(result.rm_obj_dists, result.rm_obj_labels),
              "rel_loss": F.cross_entropy(result.rel_dists, result.rel_labels[:, -1])}
    total = losses["class_loss"] + losses["rel_loss"]
    optimizer.zero_grad()
    total.backward()
    clip_grad_norm([(n, p) for n, p in detector.named_parameters() if p.grad is not None], max_norm=conf.clip, clip=True)
    optimizer.step()
    losses["total"] = total
    res = pd.Series({k: float(v) for k, v in losses.items()})
    assert set(res.index) == {"class_loss", "rel_loss", "total"} and abs(res["total"] - res["class_loss"] - res["rel_loss"]) < 1e-5
    moved = [n for n, p in detector.named_parameters() if not torch.equal(p, before[n])]
    assert moved and all(not n.startswith("detector.") for n in moved)       # the frozen detector did not move
    assert any(n.startswith("roi_fmap_obj.") for n in moved) and any(n.startswith("context.obj_ctx_rnn") for n in moved)
    scheduler.step(0.1); scheduler.step(0.1)                                 # the recipe's plateau schedule accepts it

    # what the reference's own get_optim / train_batch did to the same product surface
    for k in res.index:
        assert abs(res[k] - float(gold["train_" + k])) < 1e-5 * max(1.0, abs(res[k])), k
    assert moved == gold["train_moved"].tolist()
    np.testing.assert_allclose(param_samples(detector), gold["train_params"], rtol=1e-5, atol=1e-7)

    # the same step taken by an independent oracle model with torch's own clip + SGD gives the same loss and update
    from oracle import model as OM
    from golden.synthetic_state import CLASSES, RELS, KW
    ref = OM.RelModel(CLASSES, RELS, mode="sgcls", **KW)
    ref.load_state_dict(state); ref.train()
    for p in ref.detector.parameters():
        p.requires_grad = False
    _ones_masks(ref, B * boxes, B * boxes * (boxes - 1), B)
    ref.detector.rng = np.random.RandomState(7)
    fc = [p for n, p in ref.named_parameters() if n.startswith("roi_fmap") and p.requires_grad]
    non_fc = [p for n, p in ref.named_parameters() if not n.startswith("roi_fmap") and p.requires_grad]
    opt = torch.optim.SGD([{"params": fc, "lr": conf.lr / 10.0}, {"params": non_fc}], lr=conf.lr, momentum=0.9, weight_decay=1e-4)
    t = torch.from_numpy
    out = ref(t(nb["imgs"]), nb["im_sizes"], 0, t(nb["gt_boxes"]), t(nb["gt_classes"]), t(nb["gt_rels"]))
    loss = F.cross_entropy(out.rm_obj_dists, out.rm_obj_labels) + F.cross_entropy(out.rel_dists, out.rel_labels[:, -1])
    opt.zero_grad(); loss.backward()
    torch.nn.utils.clip_grad_norm_([p for p in ref.parameters() if p.grad is not None], 5.0)
    opt.step()
    assert abs(float(loss.detach()) - res["total"]) < 1e-5 * max(1.0, abs(res["total"]))
    want = dict(ref.named_parameters())
    for n, p in detector.named_parameters():
        assert torch.allclose(p, want[n], rtol=1e-5, atol=1e-7), n



def test_eval_rels_val_batch_runs_against_the_product():
    from config import BOX_SCALE, IM_SCALE
    from lib.evaluation.sg_eval import BasicSceneGraphEvaluator
    from dataloaders.synthetic import SyntheticBlob
    gold = np.load(GOLDEN)
    detector, nb, val, conf = eval_case()
    evaluator = BasicSceneGraphEvaluator.all_modes()
    # val_batch: one (boxes, classes, scores, rel pairs, rel scores) tuple per image with num_gpus == 1
    with torch.no_grad():
        boxes_i, objs_i, obj_scores_i, rels_i, pred_scores_i = detector[SyntheticBlob(nb, "cpu")]
    assert np.all(objs_i[rels_i[:, 0]] > 0) and np.all(objs_i[rels_i[:, 1]] > 0)
    gt_entry = {"gt_classes": val.gt_classes[0].copy(), "gt_relations": val.relationships[0].copy(),
                "gt_boxes": val.gt_boxes[0].copy()}
    e = {"pred_boxes": boxes_i * BOX_SCALE / IM_SCALE, "pred_classes": objs_i, "pred_rel_inds": rels_i,
         "obj_scores": obj_scores_i, "rel_scores": pred_scores_i}
    evaluator[conf.mode].evaluate_scene_graph_entry(gt_entry, e)
    assert e["pred_boxes"].shape == (7, 4) and e["pred_rel_inds"].shape == (42, 2) and e["rel_scores"].shape == (42, 51)
    rec = evaluator["sgcls"].result_dict["sgcls_recall"]
    assert all(len(rec[k]) == 1 and 0.0 <= rec[k][0] <= 1.0 for k in (20, 50, 100))

    # what the reference's own val_batch recorded and scored on the same product surface
    for k in ("pred_classes", "pred_rel_inds"):
        assert np.array_equal(e[k], gold["eval_" + k]), k
    for k in ("pred_boxes", "obj_scores", "rel_scores"):
        np.testing.assert_allclose(e[k], gold["eval_" + k], rtol=1e-5, atol=1e-7, err_msg=k)
    assert [rec[k][0] for k in (20, 50, 100)] == gold["eval_recall"].tolist()
