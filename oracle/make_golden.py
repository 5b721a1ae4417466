"""Generate tests/golden/*.npz FROM THE UNMODIFIED REFERENCE (test infrastructure).

Needs a checkout of the original StreamYOLO project:

    python oracle/make_golden.py REFERENCE_DIR [case ...]    # writes tests/golden/<case>.npz

It imports REFERENCE_DIR/exps/model/{yolox,dfp_pafpn,darknet,tal_head}.py untouched, on
top of the yolox==0.3.0 stand-in in oracle/ref_shim (the real package is not a
dependency of this project), loads the deterministic synthetic state_dict / frames / labels of
``streamyolo_b200.synth``, and records what the reference computes on CPU fp32:

  * train forward (model.train(), head.use_l1=True, BN eps 1e-3 / momentum 0.03 as
    cfgs/*.py:40-44): the six loss-dict values, the SimOTA assignment (foreground anchor
    ids, matched GT ids, matched IoUs), checksums of every BN running statistic after the
    step, per-BaseConv output statistics;
  * eval forward after a "calibration" train pass with momentum=1.0 (so that running
    statistics equal real batch statistics and activations stay well scaled):
    a sub-sample of the decoded [B, A, 13] output plus checksums;
  * on_pipe: first call and a buffered second call.

Importing this module (the tests take CASES from it) leaves sys.path alone apart from the
repository root; only the script run puts the original project on it.  Nothing else reads the
original project: the committed .npz files are the pin.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from streamyolo_b200 import synth  # noqa: E402

CASES = {
    # name: depth, width, H, W, B, gamma, thr, val, empty_image
    "tiny_120x160": dict(depth=0.33, width=0.125, H=120, W=160, B=2, gamma=1.0, thr=0.5, val=1.5, empty=-1),
    "tiny_empty_96x160": dict(depth=0.33, width=0.125, H=96, W=160, B=3, gamma=1.5, thr=0.4, val=1.7, empty=1),
    "s_600x960": dict(depth=0.33, width=0.50, H=600, W=960, B=2, gamma=1.0, thr=0.5, val=1.5, empty=-1),
}


def build_reference(depth, width, gamma, thr, val, momentum=0.03):
    from exps.model.dfp_pafpn import DFPPAFPN
    from exps.model.tal_head import TALHead
    from exps.model.yolox import YOLOX
    ch = [256, 512, 1024]
    model = YOLOX(DFPPAFPN(depth, width, in_channels=ch),
                  TALHead(8, width, in_channels=ch, gamma=gamma, ignore_thr=thr, ignore_value=val))
    for m in model.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.eps, m.momentum = 1e-3, momentum
    model.head.initialize_biases(1e-2)
    shapes = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    model.load_state_dict(synth.synth_state_dict(shapes), strict=True)
    model.head.use_l1 = True
    return model, shapes


def stat3(t):
    t = t.detach().double()
    return np.array([t.mean().item(), t.abs().mean().item(), t.pow(2).mean().sqrt().item()])


def capture_assignment(model):
    """Wrap dynamic_k_matching-level results without touching the reference file:
    monkey-patch get_assignments to record what it returns per image."""
    rec = []
    orig = model.head.get_assignments

    def wrapped(batch_idx, *a, **k):
        out = orig(batch_idx, *a, **k)
        gt_cls, fg_mask, pred_ious, matched, num_fg = out
        rec.append((int(batch_idx), fg_mask.nonzero()[:, 0].numpy().astype(np.int32),
                    matched.numpy().astype(np.int32), pred_ious.numpy().astype(np.float32)))
        return out
    model.head.get_assignments = wrapped
    return rec


def run_case(name, c):
    torch.manual_seed(0)
    model, shapes = build_reference(c["depth"], c["width"], c["gamma"], c["thr"], c["val"])
    x = synth.synth_frames(c["B"], c["H"], c["W"])
    fut, cur = synth.synth_labels(c["B"], c["H"], c["W"], empty_image=c["empty"])
    out = {"shape_keys": np.array(sorted(shapes)), "n_params": np.array(
        sum(p.numel() for p in model.parameters()))}

    # ---- train forward, real momentum
    conv_stats, names = {}, {}
    for n, m in model.named_modules():
        if type(m).__name__ == "BaseConv":
            m.register_forward_hook(lambda mod, i, o, n=n: conv_stats.__setitem__(n, stat3(o)))
    rec = capture_assignment(model)
    model.train()
    with torch.no_grad():
        loss = model(x, (fut, cur))
    order = ["total_loss", "iou_loss", "l1_loss", "conf_loss", "cls_loss", "num_fg"]
    out["train_loss"] = np.array([float(loss[k]) for k in order], np.float64)
    out["fg_image"] = np.concatenate([np.full(len(r[1]), r[0], np.int32) for r in rec]) if rec else np.zeros(0, np.int32)
    out["fg_anchor"] = np.concatenate([r[1] for r in rec]) if rec else np.zeros(0, np.int32)
    out["fg_gt"] = np.concatenate([r[2] for r in rec]) if rec else np.zeros(0, np.int32)
    out["fg_iou"] = np.concatenate([r[3] for r in rec]) if rec else np.zeros(0, np.float32)
    sd = model.state_dict()
    bn_keys = sorted(k for k in sd if k.endswith("running_mean") or k.endswith("running_var"))
    out["bn_keys"] = np.array(bn_keys)
    out["bn_stats_after_train"] = np.stack([stat3(sd[k]) for k in bn_keys])
    out["nbt"] = np.array([int(sd["backbone.backbone.stem.conv.bn.num_batches_tracked"]),
                           int(sd["backbone.jian2.bn.num_batches_tracked"]),
                           int(sd["head.stems.0.bn.num_batches_tracked"])])
    ck = sorted(conv_stats)
    out["conv_keys"] = np.array(ck)
    out["conv_stats_train"] = np.stack([conv_stats[k] for k in ck])

    # ---- calibration pass (momentum 1.0) then eval
    torch.manual_seed(0)
    model2, _ = build_reference(c["depth"], c["width"], c["gamma"], c["thr"], c["val"], momentum=1.0)
    # calibrate and evaluate on cat(cur, cur): both passes then see identical batch statistics,
    # so eval-mode activations reproduce the (well scaled) train-mode ones -- a well conditioned pin
    xc = torch.cat([x[:, 0:3], x[:, 0:3]], 1)
    model2.train()
    with torch.no_grad():
        model2(xc, (fut, cur))
    model2.eval()
    with torch.no_grad():
        ev = model2(xc)
    out["eval_hw"] = np.array([list(h) for h in model2.head.hw])
    sub = max(1, ev.shape[1] // 600)
    out["eval_sub_step"] = np.array(sub)
    out["eval_sub"] = ev[:, ::sub].numpy().astype(np.float32)
    out["eval_stats"] = np.stack([stat3(ev[..., j]) for j in range(ev.shape[-1])])
    # ---- on_pipe: star then buffered (dfp_pafpn.py:177-228)
    with torch.no_grad():
        o1, buf = model2(x[:1, 0:3], buffer=None, mode="on_pipe")
        o2, buf2 = model2(x[1:2, 0:3], buffer=buf, mode="on_pipe")
    out["on_pipe_stats"] = np.stack([stat3(o1), stat3(o2)] + [stat3(b) for b in buf2])
    out["on_pipe_sub2"] = o2[:, ::sub].numpy().astype(np.float32)
    path = os.path.join(ROOT, "tests", "golden", name + ".npz")
    np.savez_compressed(path, **out)
    print(name, "->", path, os.path.getsize(path) // 1024, "KiB  loss", out["train_loss"],
          "n_fg", len(out["fg_anchor"]))


def run_grad_case(name, c):
    """Backward of the reference (tools/train.py path: loss.backward(), exps/train_utils/double_trainer.py:114) on CPU
    fp32: every parameter's gradient statistics, the head prediction-conv bias gradients in full (= per-channel sums
    of d loss / d raw head output: the pin for the loss-backward kernel), and two small weight gradients in full."""
    torch.manual_seed(0)
    model, shapes = build_reference(c["depth"], c["width"], c["gamma"], c["thr"], c["val"])
    x = synth.synth_frames(c["B"], c["H"], c["W"])
    fut, cur = synth.synth_labels(c["B"], c["H"], c["W"], empty_image=c["empty"])
    model.train()
    loss = model(x, (fut, cur))
    loss["total_loss"].backward()
    out = {"total_loss": np.array(float(loss["total_loss"]), np.float64)}
    keys = [k for k, p_ in model.named_parameters() if p_.grad is not None]
    grads = dict((k, p_.grad) for k, p_ in model.named_parameters() if p_.grad is not None)
    out["grad_keys"] = np.array(keys)
    out["grad_stats"] = np.stack([stat3(grads[k]) for k in keys])
    out["grad_l2"] = np.array([float(grads[k].norm()) for k in keys], np.float64)
    for k in keys:
        if k.startswith(("head.cls_preds", "head.reg_preds", "head.obj_preds")) or k in (
                "backbone.backbone.stem.conv.bn.weight", "backbone.jian0.bn.bias", "head.stems.2.bn.weight"):
            out["g:" + k] = grads[k].numpy().astype(np.float32)
    path = os.path.join(ROOT, "tests", "golden", "grad_" + name + ".npz")
    np.savez_compressed(path, **out)
    print("grad", name, "->", path, os.path.getsize(path) // 1024, "KiB  loss", out["total_loss"], len(keys), "params")


def shapes_fixture():
    """state_dict key/shape inventory for s/m/l straight from the reference constructors."""
    inv = {}
    for tag, (d, w) in {"s": (0.33, 0.5), "m": (0.67, 0.75), "l": (1.0, 1.0)}.items():
        model, shapes = build_reference(d, w, 1.0, 0.5, 1.5)
        inv[tag + "_keys"] = np.array(list(shapes))
        inv[tag + "_shapes"] = np.array(["x".join(map(str, s)) for s in shapes.values()])
        inv[tag + "_nparams"] = np.array(sum(p.numel() for p in model.parameters()))
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "state_shapes.npz"), **inv)
    print("state_shapes:", {k: int(v) for k, v in inv.items() if k.endswith("nparams")})


if __name__ == "__main__":
    if len(sys.argv) < 2 or not os.path.isdir(os.path.join(sys.argv[1], "exps", "model")):
        sys.exit("usage: python oracle/make_golden.py REFERENCE_DIR [case ...]  (REFERENCE_DIR: a StreamYOLO checkout)")
    sys.path.insert(0, os.path.join(HERE, "ref_shim"))
    sys.path.insert(0, os.path.abspath(sys.argv[1]))
    torch.set_num_threads(os.cpu_count())
    only = sys.argv[2:]
    if not only or "shapes" in only:
        shapes_fixture()
    for n, c in CASES.items():
        if not only or n in only:
            run_case(n, c)
    for n in ("tiny_120x160", "tiny_empty_96x160"):
        if not only or "grad" in only or "grad_" + n in only:
            run_grad_case(n, CASES[n])
