"""CPU: under the overlay, the modules run_pretraining_multimae.py imports from the `multimae` package are this package's,
and the model its get_model wiring builds from them has the reference model's checkpoint schema, pinned by
tests/golden/dropin_schema.json (recorded from the reference script's own get_model by tests/golden/make_golden.py)."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCHEMA = os.path.join(ROOT, "tests", "golden", "dropin_schema.json")

# the model run_pretraining_multimae.py builds: get_model (:243-290) over DOMAIN_CONF (:49-72), from the names the script
# imports from the multimae package
BUILD = r'''
import json, sys
sys.path.insert(0, %(root)r)
import torch
from multimae_b200 import overlay
overlay.install()
import multimae_b200.multimae as mine
import multimae.multimae as mm
from multimae.criterion import MaskedCrossEntropyLoss, MaskedL1Loss, MaskedMSELoss
from multimae.input_adapters import PatchedInputAdapter, SemSegInputAdapter
from multimae.output_adapters import SpatialOutputAdapter
assert mm is mine, mm
for cls in (MaskedCrossEntropyLoss, MaskedL1Loss, MaskedMSELoss, PatchedInputAdapter, SemSegInputAdapter, SpatialOutputAdapter):
    assert cls.__module__.startswith("multimae_b200"), cls.__module__
assert torch.nn.parallel.DistributedDataParallel is overlay._IdentityDDP

with open(%(schema)r) as fh:
    ref = json.load(fh)
a = dict(ref["args"], **%(args)s)
conf = {"rgb": (PatchedInputAdapter, dict(num_channels=3), 3, 1), "depth": (PatchedInputAdapter, dict(num_channels=1), 1, 1),
        "semseg": (SemSegInputAdapter, dict(num_classes=133, dim_class_emb=64, interpolate_class_emb=False), 133, 4)}
ins = {d: conf[d][0](stride_level=conf[d][3], patch_size_full=a["patch_size"], **conf[d][1]) for d in a["in_domains"]}
def out_adapter(task):
    return SpatialOutputAdapter(num_channels=conf[task][2], stride_level=conf[task][3], patch_size_full=a["patch_size"],
                                dim_tokens=a["decoder_dim"], depth=a["decoder_depth"], num_heads=a["decoder_num_heads"],
                                use_task_queries=a["decoder_use_task_queries"], task=task, context_tasks=list(a["in_domains"]),
                                use_xattn=a["decoder_use_xattn"])
outs = {d: out_adapter(d) for d in a["out_domains"]}
if a["extra_norm_pix_loss"]:
    outs["norm_rgb"] = out_adapter("rgb")
model = getattr(mm, a["model"])(input_adapters=ins, output_adapters=outs, num_global_tokens=a["num_global_tokens"],
                                drop_path_rate=a["drop_path"])
assert type(model) is mine.MultiMAE, type(model)
'''

SCRIPT = BUILD + r'''
# checkpoint compatibility with the reference model, both directions: same keys in the same order, same shapes
sd_mine = model.state_dict()
assert [[k, list(v.shape)] for k, v in sd_mine.items()] == ref["state_dict"]
sd_ref = {k: torch.full(shape, 0.5) for k, shape in ref["state_dict"]}
model.load_state_dict(sd_ref, strict=True)
assert all(torch.equal(v, sd_ref[k]) for k, v in model.state_dict().items())
assert sorted(n for n, p in model.named_parameters() if p.requires_grad) == ref["trainable"]
assert sorted(model.no_weight_decay()) == ref["no_weight_decay"]
n = sum(p.numel() for p in model.parameters() if p.requires_grad)
assert n == ref["trainable_numel"], (n, ref["trainable_numel"])
print("DROPIN_OK", n)
'''


def test_reference_script_builds_our_model():
    res = subprocess.run([sys.executable, "-c", SCRIPT % dict(root=ROOT, schema=SCHEMA, args={})], capture_output=True,
                         text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    assert "DROPIN_OK 97917072" in res.stdout, res.stdout[-500:]


STEP_SCRIPT = r"""
import ctypes, sys
sys.path.insert(0, %(root)r)
import torch
from multimae_b200 import _lib as L
from multimae_b200 import functional as Fn

# ---- stand-ins for the GPU: a library stub that validates every call's arguments and computes nothing, zero-filled
# "uninitialised" buffers so that the losses are finite, no device synchronisation
class Stub:
    calls = []
    def __getattr__(self, name):
        res, argtypes = L.SIGNATURES[name]
        def fn(*args):
            assert len(args) == len(argtypes), name
            for a, t in zip(args, argtypes):
                if not isinstance(a, type(ctypes.byref(ctypes.c_int()))):
                    t.from_param(a)
            Stub.calls.append(name)
            return 4096 if name.endswith("_bytes") else (L.ABI_VERSION if name == "mmae_abi_version" else (b"" if name == "mmae_last_error" else 0))
        return fn
stub = Stub()
L.lib = lambda: stub
L.current_stream = lambda: 0
Fn._require_cuda = lambda t, what: None
_empty = torch.empty
torch.empty = lambda *a, **k: _empty(*a, **k).zero_()
torch.cuda.synchronize = lambda *a, **k: None
""" + BUILD + r"""
import math
from multimae_b200.native_scaler import NativeScalerWithGradNormCount
# train_one_epoch (run_pretraining_multimae.py:472-541) for two steps, as tests/test_cuda_overlay_step.py restates it
model = overlay._IdentityDDP(model)
model_without_ddp = model.module
optimizer = torch.optim.AdamW([p for p in model_without_ddp.parameters() if p.requires_grad], lr=1e-4, weight_decay=0.05,
                              betas=(0.9, 0.95), eps=1e-8)
loss_scaler = NativeScalerWithGradNormCount()
tasks_loss_fn = {"rgb": MaskedMSELoss(patch_size=16, stride=1), "depth": MaskedL1Loss(patch_size=16, stride=1),
                 "semseg": MaskedCrossEntropyLoss(patch_size=16, stride=4),
                 "norm_rgb": MaskedMSELoss(patch_size=16, stride=1, norm_pix=True)}
g = torch.Generator().manual_seed(0)
for step in range(2):
    tasks_dict = {"rgb": torch.randn(2, 3, 224, 224, generator=g), "depth": torch.rand(2, 1, 224, 224, generator=g) + 0.5,
                  "semseg": torch.randint(0, 133, (2, 56, 56), generator=g)}
    input_dict = {task: tensor for task, tensor in tasks_dict.items() if task in a["in_domains"]}
    with torch.cuda.amp.autocast():                      # :500 (no CUDA device here: a no-op)
        preds, masks = model(input_dict, num_encoded_tokens=98, alphas=1.0, sample_tasks_uniformly=False,
                             fp32_output_adapters=["semseg"])
        tasks_dict["norm_rgb"] = tasks_dict["rgb"]
        masks["norm_rgb"] = masks.get("rgb", None)
        task_losses = {task: tasks_loss_fn[task](preds[task].float(), tasks_dict[task], mask=masks.get(task, None))
                       for task in preds}
        loss = sum(task_losses.values())
    assert math.isfinite(sum(task_losses.values()).item())
    optimizer.zero_grad()
    grad_norm = loss_scaler(loss, optimizer, clip_grad=None, skip_grad=None, parameters=model.parameters(),
                            create_graph=False)
    torch.cuda.synchronize()

for name in ("mmae_sample_masks", "mmae_embed_forward", "mmae_block_forward", "mmae_ctxproj_forward", "mmae_dechead_forward_ctx",
             "mmae_dectail_forward", "mmae_masked_loss_forward", "mmae_masked_loss_backward", "mmae_dectail_backward",
             "mmae_dechead_backward_ctx", "mmae_ctxproj_backward", "mmae_block_backward", "mmae_embed_backward"):
    assert name in Stub.calls, name
# the three half-precision adapters (rgb, depth, norm_rgb) share ONE context projection GEMM and run the *_ctx heads
assert Stub.calls.count("mmae_ctxproj_forward") == 2 and Stub.calls.count("mmae_dechead_forward_ctx") == 2 * 3
assert Stub.calls.count("mmae_ctxproj_backward") == 2 and Stub.calls.count("mmae_dechead_backward_ctx") == 2 * 3
# every head's backward precedes the shared projection's backward of its step
_bw = [c for c in Stub.calls if c in ("mmae_dechead_backward_ctx", "mmae_ctxproj_backward")]
assert _bw == ["mmae_dechead_backward_ctx"] * 3 + ["mmae_ctxproj_backward"] + ["mmae_dechead_backward_ctx"] * 3 + ["mmae_ctxproj_backward"], _bw
assert "mmae_dechead_forward" not in Stub.calls and "mmae_dechead_backward" not in Stub.calls
# fp32_output_adapters=["semseg"]: that adapter's head / block / tail run through the fp32-tier entry points
# the 12 encoder blocks run chained (hand-offs fused), the one-block decoder transformers as single blocks
assert Stub.calls.count("mmae_block_forward_chain") == 2 * 12 == Stub.calls.count("mmae_block_backward_chain")
assert Stub.calls.count("mmae_block_forward") == 2 * (3 * 1) and Stub.calls.count("mmae_block_f32_forward") == 2 * 1
assert Stub.calls.count("mmae_dechead_f32_forward") == 2 and Stub.calls.count("mmae_dectail_f32_backward") == 2
assert Stub.calls.count("mmae_masked_loss_forward") == 2 * 4
assert Stub.calls.count("mmae_grad_unscale_norm") == 2                 # fused unscale + norm over the flat arena, per step
assert all(p.grad is not None and p.grad.data_ptr() == model.grad_arena().view(n).data_ptr()
           for n, p in model.named_parameters() if p.requires_grad)
print("STEP_OK", len(Stub.calls))
"""


def test_train_one_epoch_sequence_drives_our_modules():
    """The step sequence of the reference's train_one_epoch - forward with fp32_output_adapters, the four criteria,
    `optimizer.zero_grad()` after the forward, the NativeScaler call - runs two steps over the model the script builds,
    with a library stub in place of the GPU: every module-level C-ABI entry point is reached with well-formed arguments,
    in the counts the B model with one-block decoders implies."""
    res = subprocess.run([sys.executable, "-c", STEP_SCRIPT % dict(root=ROOT, schema=SCHEMA, args={"decoder_depth": 1})],
                         capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-5000:]
    assert "STEP_OK" in res.stdout, res.stdout[-500:]
