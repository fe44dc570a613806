"""Generate the golden fixtures under tests/golden/ from the LIVE reference, a checkout of EPFL-VILAB/MultiMAE named by
the environment variable MULTIMAE_REFERENCE.

    MULTIMAE_REFERENCE=/path/to/MultiMAE python tests/golden/make_golden.py

The reference (EPFL-VILAB/MultiMAE) has no tests or golden vectors of its own, so these fixtures are what pins the
oracle (oracle/multimae_oracle.py) and, through it, the CUDA path.  The reference is imported unmodified; the only
shim is a stub `torch._six` module (utils/native_scaler.py:11 imports a module removed in torch >= 2.0).

Fixtures (all fp32, CPU, torch.save of plain dicts of tensors):
  sampler_*.pt : Dirichlet shares + uniform noises fed to / index triples returned by generate_random_masks
  tiny3.pt     : 3-modality MultiMAE (dim 32, depth 2) fwd + 4 losses + all parameter gradients
  interp.pt    : RGB-only model built with the default 224 pos-emb grid run on 32x32 inputs (bicubic/bilinear resize)
  cuda_*.pt    : shapes the CUDA path supports (head_dim 64/32); weights come from tests/helpers.formula_fill_ (not
                 stored) and gradients are stored as digests (norm + strided samples)
  xtask_tiny / xout_tiny / noq_tiny / cuda_xtask / cuda_noq .pt : mask-token decoder queries (output_adapters.py:214-221) —
                 a context task left out of the call, an output task that is no context task, use_task_queries=False
  fixed_masks.pt : forward with caller-supplied task_masks (B = 1) and with mask_inputs=False: predictions
  losses.pt    : the three criteria over norm_pix / label_smoothing / mask, no mask, all-zero mask: values + prediction gradients
  depth_std.pt : truncated depth standardisation; the reference has it inline in train_one_epoch
                 (run_pretraining_multimae.py:487-492), so the statements are cut out of the reference source and executed
  dropin_schema.json : what the reference script's get_model (run_pretraining_multimae.py:243-290) builds for
                 pretrain_multimae_base with rgb+depth+semseg (+norm_rgb): state_dict keys and shapes in order, trainable
                 parameter names, no_weight_decay(), trainable parameter count

    python tests/golden/make_golden.py [fixture.pt ...]     (no names: regenerate everything)
"""
import math
import os
import sys
import types
from functools import partial

import torch

REF = os.environ.get("MULTIMAE_REFERENCE", "")
HERE = os.path.dirname(os.path.abspath(__file__))


def import_reference():
    if not os.path.isdir(REF):
        raise SystemExit("set MULTIMAE_REFERENCE to a checkout of EPFL-VILAB/MultiMAE to regenerate the fixtures")
    six = types.ModuleType("torch._six")
    six.inf = math.inf
    sys.modules.setdefault("torch._six", six)
    sys.path.insert(0, REF)
    import multimae.multimae as mm                      # noqa: E402
    from multimae.criterion import MaskedCrossEntropyLoss, MaskedL1Loss, MaskedMSELoss  # noqa: E402
    from multimae.input_adapters import PatchedInputAdapter, SemSegInputAdapter        # noqa: E402
    from multimae.output_adapters import SpatialOutputAdapter                          # noqa: E402
    return types.SimpleNamespace(mm=mm, MSE=MaskedMSELoss, L1=MaskedL1Loss, CE=MaskedCrossEntropyLoss,
                                 Patched=PatchedInputAdapter, SemSeg=SemSegInputAdapter, Spatial=SpatialOutputAdapter)


def record_sampler(R, name, B, tokens_per_task, num_encoded, alphas, seed):
    """Replays generate_random_masks' RNG consumption (multimae/multimae.py:187,195,204) to capture its draws."""
    model = R.mm.MultiMAE(input_adapters={}, output_adapters=None, dim_tokens=8, depth=0, num_heads=1)
    fake = {"t%d" % i: torch.zeros(B, n, 1) for i, n in enumerate(tokens_per_task)}
    torch.manual_seed(seed)
    masks, ids_keep, ids_restore = model.generate_random_masks(fake, num_encoded, alphas=alphas)
    torch.manual_seed(seed)
    a = [alphas] * len(tokens_per_task) if isinstance(alphas, float) else alphas
    shares = torch.distributions.Dirichlet(torch.Tensor(a)).sample((B,))
    noises = [torch.rand(B, n) for n in tokens_per_task]
    noise_all = torch.rand(B, sum(tokens_per_task))
    # sanity: the replayed draws must reproduce the recorded result through the reference formulae
    per_task = (shares * num_encoded).round().long()
    chk = []
    for i, nz in enumerate(noises):
        order = torch.argsort(nz, dim=1)
        chk.append(torch.where(order < per_task[:, i:i + 1], 0, 1))
    ids_shuffle = torch.argsort(torch.cat(chk, 1) + noise_all, dim=1)
    assert torch.equal(ids_shuffle[:, :num_encoded], ids_keep), "RNG replay diverged from the reference"
    torch.save({"shares": shares, "noises": noises, "noise_all": noise_all, "num_encoded": num_encoded,
                "task_masks": [masks[k] for k in fake], "ids_keep": ids_keep, "ids_restore": ids_restore},
               os.path.join(HERE, name))
    print("wrote", name)


def build_model(R, in_domains, dim, depth, heads, dec_dim, dec_depth, dec_heads, image_size, extra_norm_pix=True,
                out_domains=None, use_task_queries=True):
    conf = {"rgb": (3, 1), "depth": (1, 1)}
    inputs, outputs = {}, {}
    out_domains = list(in_domains) if out_domains is None else list(out_domains)
    for d in in_domains:
        if d == "semseg":
            inputs[d] = R.SemSeg(num_classes=133, dim_class_emb=64, interpolate_class_emb=False, stride_level=4,
                                 patch_size_full=16, image_size=image_size)
        else:
            inputs[d] = R.Patched(num_channels=conf[d][0], stride_level=1, patch_size_full=16, image_size=image_size)

    def out_adapter(task):
        ch, stride = (133, 4) if task == "semseg" else conf[task]
        return R.Spatial(num_channels=ch, stride_level=stride, patch_size_full=16, dim_tokens=dec_dim, depth=dec_depth,
                         num_heads=dec_heads, use_task_queries=use_task_queries, task=task,
                         context_tasks=list(in_domains), use_xattn=True, image_size=image_size)

    for d in out_domains:
        outputs[d] = out_adapter(d)
    if extra_norm_pix:
        outputs["norm_rgb"] = out_adapter("rgb")
    model = R.mm.MultiMAE(input_adapters=inputs, output_adapters=outputs, num_global_tokens=1, dim_tokens=dim,
                          depth=depth, num_heads=heads, mlp_ratio=4, qkv_bias=True,
                          norm_layer=partial(torch.nn.LayerNorm, eps=1e-6))
    # the reference leaves mask_token at zero and biases at zero; perturb so that every term is exercised
    g = torch.Generator().manual_seed(1234)
    with torch.no_grad():
        for n, p_ in model.named_parameters():
            if p_.requires_grad and (n.endswith(".bias") or n.endswith("mask_token")):
                p_.add_(torch.randn(p_.shape, generator=g) * 0.05)
    return model.float().train()


def record_model(R, name, in_domains, B, size, num_encoded, seed, formula=False, feed=None, **kw):
    """`feed`: the subset of in_domains handed to model() (train_one_epoch's input_dict); targets exist for every output
    task.  kw may carry out_domains / use_task_queries (get_model wiring, run_pretraining_multimae.py:256-283)."""
    torch.manual_seed(seed)
    model = build_model(R, in_domains, **kw)
    feed = list(in_domains) if feed is None else list(feed)
    out_domains = list(kw.get("out_domains") or in_domains)
    if formula:
        sys.path.insert(0, os.path.dirname(HERE))
        from helpers import digest, formula_fill_
        formula_fill_(list(model.named_parameters()))
    g = torch.Generator().manual_seed(seed + 1)
    x = {}
    for d in list(in_domains) + [o for o in out_domains if o not in in_domains]:
        if d == "semseg":
            x[d] = torch.randint(0, 133, (B, size // 4, size // 4), generator=g)
        else:
            x[d] = torch.randn(B, 3 if d == "rgb" else 1, size, size, generator=g)
    torch.manual_seed(seed + 2)
    tokens_like = {d: torch.zeros(B, (size // 16) ** 2, 1) for d in feed}
    triple = model.generate_random_masks(tokens_like, num_encoded, alphas=1.0)
    model.generate_random_masks = lambda *a, **k: triple          # SURVEY.md §A.5 step 3
    preds, masks = model({d: x[d] for d in feed}, num_encoded_tokens=num_encoded, alphas=1.0)
    loss_fns = {"rgb": R.MSE(16, 1), "depth": R.L1(16, 1), "semseg": R.CE(16, 4), "norm_rgb": R.MSE(16, 1, norm_pix=True)}
    losses = {}
    for task in preds:
        src = "rgb" if task == "norm_rgb" else task
        losses[task] = loss_fns[task](preds[task].float(), x[src], mask=masks.get(src))
    sum(losses.values()).backward()
    grads = {n: p_.grad.clone() for n, p_ in model.named_parameters() if p_.grad is not None}
    gnorm = torch.norm(torch.stack([g_.norm(2) for g_ in grads.values()]), 2)
    if formula:
        state, grads_out = None, {k: digest(v) for k, v in grads.items()}
    else:
        state, grads_out = {k: v.detach().clone() for k, v in model.state_dict().items()}, grads
    torch.save({
        "config": dict(in_domains=list(in_domains), B=B, size=size, num_encoded=num_encoded, formula=formula, feed=feed,
                       **kw),
        "state_dict": state,
        "inputs": x,
        "task_masks": {k: v.clone() for k, v in masks.items()},
        "ids_keep": triple[1].clone(), "ids_restore": triple[2].clone(),
        "preds": {k: v.detach().clone() for k, v in preds.items()},
        "losses": {k: v.detach().clone() for k, v in losses.items()},
        "grads": grads_out, "grad_norm": gnorm,
    }, os.path.join(HERE, name))
    print("wrote", name, {k: round(float(v), 6) for k, v in losses.items()}, "grad_norm", float(gnorm))


def record_fixed_masks(R, name):
    """MultiMAE.forward with caller-supplied task_masks (multimae/multimae.py:334-338; B = 1 like MultiMAE_Demo.ipynb) and
    with mask_inputs=False (:324-325, every token encoded): predictions only - both are invariant to the order of the kept
    tokens, which the reference's unstable argsort / random shuffle leaves open."""
    torch.manual_seed(43)
    kw = dict(dim=32, depth=2, heads=2, dec_dim=16, dec_depth=1, dec_heads=2, image_size=64)
    model = build_model(R, ("rgb", "depth", "semseg"), **kw).eval()
    g = torch.Generator().manual_seed(44)
    x1 = {"rgb": torch.randn(1, 3, 64, 64, generator=g), "depth": torch.randn(1, 1, 64, 64, generator=g),
          "semseg": torch.randint(0, 133, (1, 16, 16), generator=g)}
    tm = {k: torch.ones(1, 16, dtype=torch.long) for k in x1}
    tm["rgb"][0, [0, 5, 6, 11]] = 0
    tm["depth"][0, [3, 12]] = 0
    tm["semseg"][0, [1, 2, 8, 9, 15]] = 0
    with torch.no_grad():
        preds_fixed, masks_fixed = model(x1, task_masks=tm)
    x2 = {"rgb": torch.randn(2, 3, 64, 64, generator=g), "depth": torch.randn(2, 1, 64, 64, generator=g),
          "semseg": torch.randint(0, 133, (2, 16, 16), generator=g)}
    torch.manual_seed(45)
    with torch.no_grad():
        preds_all, masks_all = model(x2, mask_inputs=False)
    assert all(int(v.sum()) == 0 for v in masks_all.values())
    torch.save({"config": dict(in_domains=["rgb", "depth", "semseg"], **kw),
                "state_dict": {k: v.detach().clone() for k, v in model.state_dict().items()},
                "x_fixed": x1, "task_masks": tm, "preds_fixed": {k: v.clone() for k, v in preds_fixed.items()},
                "x_all": x2, "preds_all": {k: v.clone() for k, v in preds_all.items()}}, os.path.join(HERE, name))
    print("wrote", name)


def record_losses(R, name):
    """Every criterion of multimae/criterion.py over its options (norm_pix, label_smoothing, mask / no mask / all-zero
    mask / one sample without masked patches): loss value and gradient w.r.t. the prediction."""
    g = torch.Generator().manual_seed(41)
    B, S = 3, 32
    mask = (torch.rand(B, (S // 16) ** 2, generator=g) > 0.4).long()
    mask[2] = 0                                             # a sample without any masked patch (skipped by nanmean)
    mask[0, 0] = 1
    cases = {
        "mse": (R.MSE(16, 1), torch.randn(B, 3, S, S, generator=g), torch.randn(B, 3, S, S, generator=g)),
        "mse_norm_pix": (R.MSE(16, 1, norm_pix=True), torch.randn(B, 3, S, S, generator=g), torch.randn(B, 3, S, S, generator=g) * 2 + 1),
        "l1": (R.L1(16, 1), torch.randn(B, 1, S, S, generator=g), torch.randn(B, 1, S, S, generator=g)),
        "l1_norm_pix": (R.L1(16, 1, norm_pix=True), torch.randn(B, 1, S, S, generator=g), torch.randn(B, 1, S, S, generator=g) + 3),
        "ce": (R.CE(16, 4), torch.randn(B, 133, S // 4, S // 4, generator=g) * 2, torch.randint(0, 133, (B, S // 4, S // 4), generator=g)),
        "ce_smooth": (R.CE(16, 4, label_smoothing=0.1), torch.randn(B, 133, S // 4, S // 4, generator=g) * 2,
                      torch.randint(0, 133, (B, S // 4, S // 4), generator=g)),
    }
    out = {"mask": mask, "cases": {}}
    for key, (fn, pred, tgt) in cases.items():
        rec = {"pred": pred, "target": tgt}
        for mname, m in (("masked", mask), ("none", None), ("zero", torch.zeros_like(mask))):
            pr = pred.clone().requires_grad_(True)
            loss = fn(pr, tgt, mask=m)
            rec["loss_" + mname] = loss.detach().clone().float()
            if loss.requires_grad:
                loss.backward()
                rec["grad_" + mname] = pr.grad.clone()
        out["cases"][key] = rec
    torch.save(out, os.path.join(HERE, name))
    print("wrote", name, {k: round(float(v["loss_masked"]), 6) for k, v in out["cases"].items()})


def record_dropin_schema(name):
    """The model the reference script's own get_model builds from the arguments of a default pre-training run."""
    import json
    sys.path.insert(0, REF)
    import run_pretraining_multimae as script          # noqa: E402
    args = types.SimpleNamespace(model="pretrain_multimae_base", in_domains=["rgb", "depth", "semseg"],
                                 out_domains=["rgb", "depth", "semseg"], patch_size=16, decoder_dim=256, decoder_depth=2,
                                 decoder_num_heads=8, decoder_use_task_queries=True, decoder_use_xattn=True,
                                 extra_norm_pix_loss=True, num_global_tokens=1, drop_path=0.0)
    model = script.get_model(args)
    out = {"args": vars(args),
           "state_dict": [[k, list(v.shape)] for k, v in model.state_dict().items()],
           "trainable": sorted(n for n, p_ in model.named_parameters() if p_.requires_grad),
           "no_weight_decay": sorted(model.no_weight_decay()),
           "trainable_numel": sum(p_.numel() for p_ in model.parameters() if p_.requires_grad)}
    with open(os.path.join(HERE, name), "w") as fh:              # one entry per line
        fh.write("{\n" + ",\n".join("%s: %s" % (json.dumps(k), json.dumps(v) if k != "state_dict" else
                                                 "[\n" + ",\n".join(json.dumps(e) for e in v) + "\n]")
                                     for k, v in out.items()) + "\n}\n")
    print("wrote", name, "(%d state_dict entries)" % len(out["state_dict"]))


def record_depth_standardize(name):
    """Executes the reference's OWN statements (the body of `if standardize_depth and 'depth' in tasks_dict:` in
    train_one_epoch, run_pretraining_multimae.py:487-492) on synthetic depth maps and records input and result."""
    import textwrap
    from einops import rearrange
    src = open(os.path.join(REF, "run_pretraining_multimae.py")).read().splitlines()
    start = next(i for i, ln in enumerate(src) if "if standardize_depth and 'depth' in tasks_dict" in ln)
    body = []
    for ln in src[start + 1:]:
        if ln.strip() and (len(ln) - len(ln.lstrip())) <= (len(src[start]) - len(src[start].lstrip())):
            break
        body.append(ln)
    code = textwrap.dedent("\n".join(body))
    assert "torch.sort" in code and "trunc_depth.var" in code, code
    g = torch.Generator().manual_seed(31)
    depth = torch.randn(4, 1, 24, 24, generator=g)
    depth[1] = depth[1].abs() * 3 + 0.5                                   # metric-depth-like: positive, skewed
    depth[2] = torch.round(depth[2] * 2) / 2                              # heavy ties, also across the 10 % / 90 % cuts
    depth[3, :, :12] = 7.25                                               # one value covering half of the map
    ns = {"torch": torch, "rearrange": rearrange, "tasks_dict": {"depth": depth.clone()}}
    exec(code, ns)
    torch.save({"depth": depth, "standardized": ns["tasks_dict"]["depth"].clone()},
               os.path.join(HERE, name))
    print("wrote", name, "(executed %d reference source lines)" % len(code.splitlines()))


if __name__ == "__main__":
    only = set(sys.argv[1:])
    if only == {"depth_std.pt"}:
        if not os.path.isdir(REF):
            raise SystemExit("set MULTIMAE_REFERENCE to a checkout of EPFL-VILAB/MultiMAE")
        record_depth_standardize("depth_std.pt")
        raise SystemExit(0)
    if only == {"dropin_schema.json"}:
        import_reference()
        record_dropin_schema("dropin_schema.json")
        raise SystemExit(0)
    R = import_reference()
    # mask-token queries (multimae/output_adapters.py:214-221): a task that is reconstructed without being fed
    # (its embedding exists: context task left out of this call / does not exist: not a context task), and
    # --decoder_use_task_queries False
    xtask = dict(
        xtask_tiny=lambda: record_model(R, "xtask_tiny.pt", ("rgb", "depth", "semseg"), B=3, size=64, num_encoded=10, seed=31,
                                        feed=("rgb", "semseg"), dim=32, depth=2, heads=2, dec_dim=16, dec_depth=1,
                                        dec_heads=2, image_size=64),
        xout_tiny=lambda: record_model(R, "xout_tiny.pt", ("rgb",), B=2, size=64, num_encoded=6, seed=33,
                                       out_domains=("rgb", "depth"), dim=32, depth=1, heads=2, dec_dim=16, dec_depth=1,
                                       dec_heads=2, image_size=64),
        noq_tiny=lambda: record_model(R, "noq_tiny.pt", ("rgb", "depth"), B=2, size=64, num_encoded=8, seed=35,
                                      use_task_queries=False, dim=32, depth=1, heads=2, dec_dim=16, dec_depth=1,
                                      dec_heads=2, image_size=64),
        cuda_xtask=lambda: record_model(R, "cuda_xtask.pt", ("rgb", "depth", "semseg"), B=2, size=64, num_encoded=10, seed=37,
                                        formula=True, feed=("rgb", "semseg"), dim=128, depth=1, heads=2, dec_dim=128,
                                        dec_depth=1, dec_heads=4, image_size=64),
        cuda_noq=lambda: record_model(R, "cuda_noq.pt", ("rgb", "depth"), B=2, size=64, num_encoded=8, seed=39, formula=True,
                                      use_task_queries=False, out_domains=("rgb", "depth", "semseg"), dim=128, depth=1,
                                      heads=2, dec_dim=128, dec_depth=1, dec_heads=4, image_size=64),
    )
    if only == {"fixed_masks.pt"}:
        record_fixed_masks(R, "fixed_masks.pt")
        raise SystemExit(0)
    if only == {"losses.pt"}:
        record_losses(R, "losses.pt")
        raise SystemExit(0)
    if only and only <= {k + ".pt" for k in xtask}:
        for k, fn in xtask.items():
            if k + ".pt" in only:
                fn()
        raise SystemExit(0)
    for fn in xtask.values():
        fn()
    record_losses(R, "losses.pt")
    record_fixed_masks(R, "fixed_masks.pt")
    record_depth_standardize("depth_std.pt")
    record_dropin_schema("dropin_schema.json")
    record_sampler(R, "sampler_small.pt", B=16, tokens_per_task=[16, 16, 16], num_encoded=12, alphas=1.0, seed=3)
    record_sampler(R, "sampler_cfg2.pt", B=8, tokens_per_task=[196, 196, 196], num_encoded=98, alphas=1.0, seed=4)
    record_sampler(R, "sampler_alpha.pt", B=8, tokens_per_task=[196, 196], num_encoded=98, alphas=[0.5, 2.0], seed=5)
    record_model(R, "tiny3.pt", ("rgb", "depth", "semseg"), B=3, size=64, num_encoded=12, seed=7,
                 dim=32, depth=2, heads=2, dec_dim=16, dec_depth=1, dec_heads=2, image_size=64)
    record_model(R, "interp.pt", ("rgb",), B=2, size=32, num_encoded=2, seed=11,
                 dim=32, depth=1, heads=2, dec_dim=16, dec_depth=1, dec_heads=2, image_size=224)
    # CUDA-runnable shapes (head_dim 64 / 32, widths multiple of 128); weights from tests/helpers.formula_fill_
    record_model(R, "cuda_small.pt", ("rgb", "depth", "semseg"), B=3, size=64, num_encoded=12, seed=21, formula=True,
                 dim=128, depth=2, heads=2, dec_dim=128, dec_depth=1, dec_heads=4, image_size=64)
    record_model(R, "cuda_interp.pt", ("rgb", "semseg"), B=2, size=96, num_encoded=20, seed=23, formula=True,
                 dim=128, depth=1, heads=2, dec_dim=128, dec_depth=1, dec_heads=4, image_size=224)
