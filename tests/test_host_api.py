"""CPU: host-side contract of the drop-in modules (no kernel is executed here).

 * the C-ABI library loads and exports every symbol include/multimae_b200.h declares;
 * module constructors / parameter names / shapes follow the reference state_dict schema (SURVEY.md §A.1);
 * the product path refuses to run without CUDA (no CPU fallback)."""
import os
import re
import subprocess
import sys

import pytest
import torch

from oracle import multimae_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _build(in_domains=("rgb", "depth", "semseg"), dim=128, depth=2, heads=2, dec_dim=128, dec_depth=1, dec_heads=4,
           image_size=64, out_domains=None, use_task_queries=True):
    from multimae_b200.input_adapters import PatchedInputAdapter, SemSegInputAdapter
    from multimae_b200.multimae import MultiMAE
    from multimae_b200.output_adapters import SpatialOutputAdapter
    conf = {"rgb": (3, 1), "depth": (1, 1), "semseg": (133, 4)}
    ins, outs = {}, {}
    for d in in_domains:
        if d == "semseg":
            ins[d] = SemSegInputAdapter(num_classes=133, dim_class_emb=64, stride_level=4, patch_size_full=16,
                                        image_size=image_size)
        else:
            ins[d] = PatchedInputAdapter(num_channels=conf[d][0], stride_level=1, patch_size_full=16, image_size=image_size)
    for key in list(in_domains if out_domains is None else out_domains) + ["norm_rgb"]:
        task = "rgb" if key == "norm_rgb" else key
        ch, stride = conf[task]
        outs[key] = SpatialOutputAdapter(num_channels=ch, stride_level=stride, patch_size_full=16, dim_tokens=dec_dim,
                                         depth=dec_depth, num_heads=dec_heads, task=task, context_tasks=list(in_domains),
                                         image_size=image_size, use_task_queries=use_task_queries)
    return MultiMAE(ins, outs, num_global_tokens=1, dim_tokens=dim, depth=depth, num_heads=heads)


def test_abi_exports_every_declared_symbol():
    from multimae_b200 import _lib as L
    from multimae_b200.build import build
    build()
    handle = L.lib()
    header = open(os.path.join(ROOT, "include", "multimae_b200.h")).read()
    declared = set(re.findall(r"\b(mmae_[a-z0-9_]+)\s*\(", header))
    assert declared == set(L.SIGNATURES), (declared ^ set(L.SIGNATURES))
    for name in declared:
        assert getattr(handle, name) is not None
    assert handle.mmae_abi_version() == L.ABI_VERSION
    # loading the library launches nothing; counted in a fresh process, since GPU tests of this session add to the counter
    res = subprocess.run([sys.executable, "-c", "import sys; sys.path.insert(0, %r); from multimae_b200 import _lib as L; "
                          "print(L.lib().mmae_launch_count())" % ROOT], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0 and res.stdout.split() == ["0"], res.stdout[-500:] + res.stderr[-2000:]


def test_state_dict_schema_and_roundtrip(golden_dir):
    fx = torch.load(os.path.join(golden_dir, "cuda_small.pt"), map_location="cpu", weights_only=False)
    c = fx["config"]
    model = _build(tuple(c["in_domains"]), c["dim"], c["depth"], c["heads"], c["dec_dim"], c["dec_depth"], c["dec_heads"],
                   c["image_size"])
    cfg = O.make_config(in_domains=tuple(c["in_domains"]))
    cfg.dim, cfg.depth, cfg.heads = c["dim"], c["depth"], c["heads"]
    cfg.dec_dim, cfg.dec_depth, cfg.dec_heads = c["dec_dim"], c["dec_depth"], c["dec_heads"]
    cfg.posemb_grid = c["image_size"] // 16
    ref = O.init_params(cfg)                       # schema pinned to the reference by test_oracle_golden
    sd = model.state_dict()
    assert set(sd) == set(ref)
    for k, v in ref.items():
        assert tuple(sd[k].shape) == tuple(v.shape), k
    for k in sd:
        if k.endswith("pos_emb"):
            torch.testing.assert_close(sd[k], ref[k], rtol=0, atol=1e-6)
    assert {k for k, p in model.named_parameters() if not p.requires_grad} == {k for k in ref if k.endswith("pos_emb")}
    model.load_state_dict(ref, strict=True)          # reference-schema checkpoint loads strictly
    assert "global_tokens" in model.no_weight_decay()
    assert "input_adapters.semseg.class_emb" in model.no_weight_decay()


def test_full_size_parameter_count():
    from multimae_b200.input_adapters import PatchedInputAdapter, SemSegInputAdapter
    from multimae_b200.multimae import pretrain_multimae_base
    from multimae_b200.output_adapters import SpatialOutputAdapter
    ins = {"rgb": PatchedInputAdapter(3, 1, 16), "depth": PatchedInputAdapter(1, 1, 16),
           "semseg": SemSegInputAdapter(133, 4, 16, dim_class_emb=64)}
    outs = {}
    for key, (ch, st, task) in {"rgb": (3, 1, "rgb"), "depth": (1, 1, "depth"), "semseg": (133, 4, "semseg"),
                                "norm_rgb": (3, 1, "rgb")}.items():
        outs[key] = SpatialOutputAdapter(ch, st, 16, dim_tokens=256, depth=2, num_heads=8, task=task,
                                         context_tasks=["rgb", "depth", "semseg"])
    model = pretrain_multimae_base(ins, outs, num_global_tokens=1, drop_path_rate=0.0)
    trainable = sum(p.numel() for p in model.parameters() if p.requires_grad)
    assert trainable == 97_917_632 or abs(trainable - 97.92e6) < 0.01e6, trainable      # SURVEY.md §0: 97.92 M
    assert model.get_num_layers() == 12


def test_no_cpu_fallback():
    from multimae_b200 import _lib as L
    from multimae_b200.criterion import MaskedMSELoss
    model = _build()
    x = {"rgb": torch.randn(1, 3, 64, 64), "depth": torch.randn(1, 1, 64, 64),
         "semseg": torch.randint(0, 133, (1, 16, 16))}
    with pytest.raises(L.MmaeError):
        model(x, num_encoded_tokens=12)
    with pytest.raises(L.MmaeError):
        MaskedMSELoss()(torch.randn(1, 3, 32, 32), torch.randn(1, 3, 32, 32))
    from multimae_b200.functional import standardize_depth
    with pytest.raises(L.MmaeError):
        standardize_depth(torch.randn(2, 1, 16, 16))


def test_grad_arena_layout():
    from multimae_b200.functional import GradArena
    model = _build()
    named = [(n, p) for n, p in model.named_parameters() if p.requires_grad]
    arena = GradArena(named, torch.device("cpu"))
    assert arena.numel >= sum(p.numel() for _, p in named)
    for n, p in named:
        v = arena.view(n)
        assert v.shape == p.shape and v.data_ptr() % 16 == 0
    arena.flat.fill_(1.0)
    arena.zero_()
    assert float(arena.flat.abs().sum()) == 0.0


def test_ctypes_structs_match_the_c_header(tmp_path):
    """Every struct of include/multimae_b200.h against its ctypes twin in multimae_b200/_lib.py: sizeof and the offset of
    every field, as a C compiler lays them out (gcc on the header itself - the header is plain C)."""
    import ctypes
    import shutil
    import subprocess
    from multimae_b200 import _lib as L
    gcc = shutil.which("gcc") or shutil.which("cc")
    if gcc is None:
        pytest.skip("no C compiler")
    pairs = {"mmae_gemm_epilogue": L.GemmEpilogue, "mmae_embed_layout": L.EmbedLayout, "mmae_embed_inputs": L.EmbedInputs,
             "mmae_embed_params": L.EmbedParams, "mmae_embed_grads": L.EmbedGrads, "mmae_block_params": L.BlockParams,
             "mmae_block_grads": L.BlockGrads, "mmae_decoder_index": L.DecoderIndex, "mmae_dechead_params": L.DecHeadParams,
             "mmae_dechead_grads": L.DecHeadGrads, "mmae_ctxproj_params": L.CtxProjParams, "mmae_ctxproj_grads": L.CtxProjGrads}
    header = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "multimae_b200.h")
    declared = set(re.findall(r"^\} (mmae_\w+);", open(header).read(), re.M))
    assert declared == set(pairs), declared ^ set(pairs)
    lines = ["#include <stdio.h>", "#include <stddef.h>", '#include "%s"' % header, "int main(void) {"]
    for cname, cls in pairs.items():
        lines.append('  printf("%s sizeof %%zu\\n", sizeof(%s));' % (cname, cname))
        for fname, _ in cls._fields_:
            lines.append('  printf("%s %s %%zu\\n", offsetof(%s, %s));' % (cname, fname, cname, fname))
    lines += ["  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run([gcc, "-std=c99", "-o", str(exe), str(src)], check=True, capture_output=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout
    for line in out.strip().splitlines():
        cname, field, value = line.split()
        cls = pairs[cname]
        mine = ctypes.sizeof(cls) if field == "sizeof" else getattr(cls, field).offset
        assert mine == int(value), "%s.%s: ctypes %d, C %s" % (cname, field, mine, value)
    assert L.MAX_TASKS == int(re.search(r"#define MMAE_MAX_TASKS (\d+)", open(header).read()).group(1))
    assert L.ABI_VERSION == int(re.search(r"#define MMAE_ABI_VERSION (\d+)", open(header).read()).group(1))


def test_c_abi_rejects_bad_arguments_before_any_launch():
    """Error behaviour of the C ABI (no GPU needed: every check fires before the first CUDA call): a non-zero code,
    the message behind mmae_last_error(), and the Python stub's exception (MmaeError, a RuntimeError like the reference's
    assertion failures, e.g. multimae/input_adapters.py:105-106)."""
    import ctypes
    from multimae_b200 import _lib as L
    lib = L.lib()
    ep = L.GemmEpilogue()
    ARG, UNSUPPORTED = 1, 3
    cases = [
        (lib.mmae_gemm_bf16(None, 0, 0, None, 0, 0, 128, 128, 64, 1, ctypes.byref(ep), None), ARG, b"null operand"),
        (lib.mmae_gemm_bf16(16, 64, 0, 16, 64, 0, 128, 100, 64, 1, ctypes.byref(ep), None), ARG, b"multiple of 8"),
        (lib.mmae_standardize_depth(None, None, 1, 16, 1, 9, 1e-6, None, None), ARG, b"bad args"),
        (lib.mmae_standardize_depth(16, 16, 1, 16, 9, 9, 1e-6, None, None), ARG, b"lo < hi"),
        (lib.mmae_standardize_depth_set_variant(3), ARG, b"1 or 2"),
        (lib.mmae_layernorm_forward(16, 100, 16, 16, 16, 100, None, 0, 16, 16, 4, 100, 1e-6, None), UNSUPPORTED, b"multiple of 128"),
        (lib.mmae_attention_forward(16, 64, 16, 64, 16, 64, 16, 64, None, 1, 1, 8, 8, 48, 0.1, None), UNSUPPORTED, b"head_dim 48"),
        (lib.mmae_masked_loss_forward(5, 0, 0.0, 16, 16, None, 1, 3, 32, 32, 16, 16, 16, None), UNSUPPORTED, b"kind"),
    ]
    # round-2 entry points: shared context projection, *_ctx heads, chained blocks
    cp = L.CtxProjParams()
    cp.num = 2
    cp.dim[0], cp.dim[1] = 256, 100                                      # 100 is not a multiple of 8
    cp.weight[0] = cp.weight[1] = cp.bias[0] = cp.bias[1] = 16
    bp, bg = L.BlockParams(), L.BlockGrads()
    cases += [
        (lib.mmae_ctxproj_forward(16, 128, 768, ctypes.byref(cp), 16, 16, None), ARG, b"mmae_ctxproj_forward"),
        (lib.mmae_ctxproj_forward(None, 128, 768, ctypes.byref(cp), 16, 16, None), ARG, b"mmae_ctxproj_forward"),
        (lib.mmae_ctxproj_backward(128, 768, ctypes.byref(cp), ctypes.byref(L.CtxProjGrads()), None, 16, 16, None), ARG,
         b"mmae_ctxproj_backward"),
        (lib.mmae_dechead_forward_ctx(None, 1024, None, 8, 1024, 1e-6, None, None, None, None, None), ARG, b"bad args"),
        (lib.mmae_dechead_backward_ctx(None, 8, 1024, None, None, None, None, 1024, None, None, None), ARG, b"bad args"),
        # x_add without a buffer for the sum; neither x_out nor y_out; a bf16 gradient copy without its column-sum target
        (lib.mmae_block_forward_chain(16, 16, None, 16, None, 2, 8, 128, 2, 512, 1e-6, ctypes.byref(bp), 16, 16, None), ARG,
         b"mmae_block_forward"),
        (lib.mmae_block_forward_chain(16, None, None, None, None, 2, 8, 128, 2, 512, 1e-6, ctypes.byref(bp), 16, 16, None), ARG,
         b"mmae_block_forward"),
        (lib.mmae_block_backward_chain(16, 16, None, 16, 16, None, 2, 8, 128, 2, 512, ctypes.byref(bp), ctypes.byref(bg), 16,
                                       16, None), ARG, b"mmae_block_backward"),
    ]
    assert lib.mmae_block_saved_x_mid(None, 2, 8, 128, 2, 512) is None
    # mmae_last_error() holds the message of the most recent failure: re-issue each call to read its own message
    assert [rc for rc, _, _ in cases] == [want for _, want, _ in cases]
    assert lib.mmae_gemm_bf16(16, 64, 0, 16, 64, 0, 128, 100, 64, 1, ctypes.byref(ep), None) == ARG
    assert b"N=100 must be a multiple of 8" in lib.mmae_last_error()
    with pytest.raises(L.MmaeError, match="multiple of 8"):
        L.check(lib.mmae_gemm_bf16(16, 64, 0, 16, 64, 0, 128, 100, 64, 1, ctypes.byref(ep), None), "mmae_gemm_bf16")
    assert issubclass(L.MmaeError, RuntimeError)
    assert lib.mmae_standardize_depth_set_variant(1) == 0


def test_product_never_touches_the_oracle_or_the_reference():
    """The oracle is test infrastructure: nothing under multimae_b200/ (Python or CUDA sources) may import, load or name it,
    nor read /root/reference; importing the whole package must not pull `oracle` into sys.modules."""
    import subprocess
    import sys
    pkg = os.path.join(ROOT, "multimae_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, re.M), f
                assert "multimae_oracle" not in text and "/root/reference" not in text, f
    code = ("import sys; sys.path.insert(0, %r); import multimae_b200.multimae, multimae_b200.criterion, multimae_b200.optim, "
            "multimae_b200.parallel, multimae_b200.train_step, multimae_b200.native_scaler, multimae_b200.overlay, "
            "multimae_b200.kernels; assert not [m for m in sys.modules if m == 'oracle' or m.startswith('oracle.')]; print('ok')" % ROOT)
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0 and "ok" in res.stdout, res.stderr[-2000:]
