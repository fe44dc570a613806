"""bench.py — MultiMAE-B pre-training step throughput on B200 (BASELINE.json metric).

    python bench.py --gpus 1 --steps 20 --warmup 5                      # this framework (CUDA path)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 ... bench.py --gpus 8 --steps K --warmup W
    python bench.py --impl reference --gpus 1 --steps 3 --warmup 1      # CPU arm: the oracle port on the host cores

Workload (config.workload): BASELINE.json configs[1] — MultiMAE-B, rgb+depth+semseg in/out + norm_rgb decoder, 224x224,
98 visible tokens, bs=128 per GPU, bf16 tensor-core operands / fp32 accumulate; data-parallel for N>1 (weak scaling).
One step = forward + 4 masked losses + backward + bucketed gradient all-reduce (N>1) + fused unscale/grad-norm + AdamW.
Prints ONE JSON line on rank 0.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ALG_FLOP_PER_SAMPLE = 65.41e9        # fwd+bwd, algorithmic (BASELINE.md §3, SURVEY.md §8d)
METRIC = "MultiMAE-B pretrain samples/sec @ bs=128/GPU"
WORKLOAD = "MultiMAE-B rgb+depth+semseg(+norm_rgb) 224x224, 98 visible tokens, bs=128/GPU, fwd+4 losses+bwd+allreduce+AdamW"
# --workload: the default is the configuration BASELINE.json's metric is quoted on (configs[1] / [2]); configs[3] and [4]
# are its per-GPU stress cases (algorithmic FLOP per sample: SURVEY.md §8d table)
WORKLOADS = {
    "cfg2": dict(size="base", image=224, visible=98, batch=128, flop=ALG_FLOP_PER_SAMPLE, metric=METRIC, name=WORKLOAD),
    "cfg4": dict(size="large", image=224, visible=98, batch=64, flop=196.40e9,
                 metric="MultiMAE-L pretrain samples/sec @ bs=64/GPU",
                 name="MultiMAE-L (24 layers, d=1024, 16 heads) rgb+depth+semseg(+norm_rgb) 224x224, 98 visible tokens, "
                      "bs=64/GPU, fwd+4 losses+bwd+allreduce+AdamW"),
    "cfg5": dict(size="base", image=448, visible=392, batch=32, flop=287.0e9,
                 metric="MultiMAE-B 448x448 pretrain samples/sec @ bs=32/GPU",
                 name="MultiMAE-B rgb+depth+semseg(+norm_rgb) 448x448 (784 patches/modality, 392 visible tokens), bs=32/GPU, "
                      "fwd+4 losses+bwd+allreduce+AdamW"),
}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1590.0)), d.get("hbm_gbs", 6650.0), "measured"
    return 1400.0, 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.proc, self.idx = None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms",
                                          "100", "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                                         text=True)
        except Exception:  # noqa: BLE001
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        for line in out.strip().splitlines():
            f = [t.strip() for t in line.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def build_model_and_losses(device, size="base", image=224):
    from multimae_b200.criterion import MaskedCrossEntropyLoss, MaskedL1Loss, MaskedMSELoss
    from multimae_b200.input_adapters import PatchedInputAdapter, SemSegInputAdapter
    from multimae_b200.multimae import pretrain_multimae_base, pretrain_multimae_large
    from multimae_b200.output_adapters import SpatialOutputAdapter
    doms = ["rgb", "depth", "semseg"]
    # like get_model (run_pretraining_multimae.py:248-283) the adapters keep their default image_size=224: at 448^2 inputs
    # the 14x14 sin-cos tables are resized to 28x28 (bicubic / bilinear) - once, the resized table is cached
    del image
    ins = {"rgb": PatchedInputAdapter(num_channels=3, stride_level=1, patch_size_full=16),
           "depth": PatchedInputAdapter(num_channels=1, stride_level=1, patch_size_full=16),
           "semseg": SemSegInputAdapter(num_classes=133, dim_class_emb=64, interpolate_class_emb=False, stride_level=4,
                                        patch_size_full=16)}
    outs = {}
    for key, (ch, stride, task) in {"rgb": (3, 1, "rgb"), "depth": (1, 1, "depth"), "semseg": (133, 4, "semseg"),
                                    "norm_rgb": (3, 1, "rgb")}.items():
        outs[key] = SpatialOutputAdapter(num_channels=ch, stride_level=stride, patch_size_full=16, dim_tokens=256, depth=2,
                                         num_heads=8, use_task_queries=True, task=task, context_tasks=doms, use_xattn=True)
    factory = pretrain_multimae_base if size == "base" else pretrain_multimae_large
    model = factory(ins, outs, num_global_tokens=1, drop_path_rate=0.0).to(device).train()
    losses = {"rgb": MaskedMSELoss(16, 1), "depth": MaskedL1Loss(16, 1), "semseg": MaskedCrossEntropyLoss(16, 4),
              "norm_rgb": MaskedMSELoss(16, 1, norm_pix=True)}
    return model, losses


_T0 = time.perf_counter()


_JSON_FD = None


def _quiet_stdout():
    """Point fd 1 at stderr for the duration of the run: native libraries write banners to it (NCCL prints its version
    line there when the first communicator is built) and the contract is ONE JSON line on stdout.  _emit() restores it."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def _emit(obj):
    sys.stdout.flush()
    if _JSON_FD is not None:
        os.dup2(_JSON_FD, 1)
    print(json.dumps(obj), flush=True)


def _note(msg):
    """progress on stderr (the JSON line on stdout stays the only stdout output)"""
    print("[bench %6.1fs] %s" % (time.perf_counter() - _T0, msg), file=sys.stderr, flush=True)


def ncu_evidence():
    """Figures that only a profiler can give (DRAM bytes of the dominant GEMM, tensor-pipe % of the attention kernels) are
    READ from the committed summary of the `ncu --set full` capture - profiles/ncu_hot_kernels.json, written by
    scripts/ncu_raw_table.py --json together with the commit it was taken at - never typed into this file."""
    path = os.path.join(ROOT, "profiles", "ncu_hot_kernels.json")
    try:
        with open(path) as fh:
            return json.load(fh)
    except Exception:  # noqa: BLE001
        return None


def encoder_tc_from_table(agg, rows_enc, D_enc, peak_tf):
    """BASELINE metric, second half ("encoder TC util%").  `agg`: {(M, N, K, operand-major flags, split): [launches, ms]}
    of one profiled step.  The GEMMs of the encoder blocks (QKV, proj, fc1, fc2; forward, dgrad, wgrad) are the launches
    whose three extents are the encoder row count B*(visible+1) and two of {D, 3D, 4D}; their FLOPs over their CUDA-event
    time, against the measured and the nominal dense bf16 peak."""
    widths = {D_enc, 3 * D_enc, 4 * D_enc}
    fl_enc = ms_enc = 0.0
    n_enc = 0
    for (M_, N_, K_, _maj, _split), (cnt, ms_) in agg.items():
        dims = [M_, N_, K_]
        if rows_enc not in dims:
            continue
        dims.remove(rows_enc)
        if dims[0] in widths and dims[1] in widths:
            fl_enc += 2.0 * M_ * N_ * K_ * cnt
            ms_enc += ms_
            n_enc += cnt
    if ms_enc <= 0:
        return None
    tf_enc = fl_enc / (ms_enc * 1e-3) / 1e12
    out = {"encoder_gemm_tflops": round(tf_enc, 1), "launches_per_step": n_enc, "ms_per_step": round(ms_enc, 3),
           "frac_of_measured_peak": round(tf_enc / peak_tf, 4), "frac_of_nominal_2250": round(tf_enc / 2250.0, 4)}
    ev = ncu_evidence()
    if ev is not None:
        out["tensor_pipe_pct_ncu"] = {k: v.get("tensor_pct") for k, v in ev.get("kernels", {}).items()
                                      if "attn" in k or "gemm" in k}
        out["ncu_capture"] = {"file": "profiles/ncu_hot_kernels.json", "commit": ev.get("commit"), "when": ev.get("when")}
    return out


def synthetic_batch(B, seed, pin=False, image=224):
    g = torch.Generator().manual_seed(seed)
    x = {"rgb": torch.randn(B, 3, image, image, generator=g), "depth": torch.randn(B, 1, image, image, generator=g),
         "semseg": torch.randint(0, 133, (B, image // 4, image // 4), generator=g)}
    return {k: v.pin_memory() for k, v in x.items()} if pin else x


DUMP_SAMPLE = 1 << 20        # parameter / gradient values kept by --dump-outputs (4 MB each in float32)


def optimizer_state(opt, clone=False):
    """Parameters, Adam moments and the device {lr, step} scalars: everything a training step reads besides its batch."""
    state = (opt.flat_params, opt.exp_avg, opt.exp_avg_sq, opt._dyn)
    return tuple(t.clone() for t in state) if clone else state


def dump_outputs(out_dir, model, opt, loss, grad_norm):
    """What one step computed, as DIR/<name>.npy: the loss and gradient norm the step returns, and the same fixed, seeded
    sample of the updated parameters and of the gradients it left in the arena (trainable parameters in
    named_parameters() order, padding between the arena's slots excluded)."""
    import numpy as np
    arena = model.grad_arena()
    named = [n for n, p in model.named_parameters() if p.requires_grad]
    params = torch.cat([opt.flat_params[arena.offsets[n][0]:arena.offsets[n][0] + arena.offsets[n][1]] for n in named])
    grads = torch.cat([arena.flat[arena.offsets[n][0]:arena.offsets[n][0] + arena.offsets[n][1]] for n in named])
    idx = torch.randint(0, params.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values
    idx = idx.to(params.device)
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": loss.detach().reshape(1), "grad_norm": grad_norm.detach().reshape(1),
              "params_sample": params[idx], "grads_sample": grads[idx]}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())
    _note("wrote %s to %s" % (", ".join(n + ".npy" for n in arrays), out_dir))


def run_ours(args, rank, world, local_rank):
    import torch.distributed as dist
    from multimae_b200 import _lib as L
    from multimae_b200.native_scaler import NativeScalerWithGradNormCount
    from multimae_b200.optim import FlatAdamW
    from multimae_b200.parallel import attach_data_parallel, broadcast_parameters

    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    torch.manual_seed(0)                                   # identical init on every rank
    wl = WORKLOADS[args.workload]
    model, loss_fns = build_model_and_losses(device, wl["size"], wl["image"])
    broadcast_parameters(model)
    opt = FlatAdamW(model, lr=1e-4 * args.batch * world / 256, betas=(0.9, 0.95), weight_decay=0.05)
    # bf16 operands keep fp32's exponent range: no loss scaling needed (the reference's GradScaler exists for fp16)
    scaler = NativeScalerWithGradNormCount(enabled=False).attach_arena(model.grad_arena())
    if world > 1:
        attach_data_parallel(model, scaler)
    initial_state = optimizer_state(opt, clone=True) if args.dump_outputs else None
    torch.manual_seed(1234 + rank)                         # per-rank data / masks (run_pretraining_multimae.py:300)
    B = args.batch
    host = [synthetic_batch(B, 100 * rank + i, pin=True, image=wl["image"]) for i in range(2)]   # 2 x 106 MB: > L2 together
    resident = [{k: v.to(device) for k, v in hb.items()} for hb in host]
    lib = L.lib()

    from multimae_b200.train_step import TrainStep
    stepper = TrainStep(model, loss_fns, opt, scaler, num_encoded_tokens=wl["visible"], alphas=1.0,
                        loss_sources={"norm_rgb": "rgb"}, standardize_depth=bool(args.standardize_depth))
    if world > 1:
        # the first collectives build NCCL's channels / buffers: keep that out of every timed region
        for _ in range(3):
            dist.all_reduce(model.grad_arena().flat)
        model.grad_arena().zero_()
        torch.cuda.synchronize()
        if args.sm_budget:
            lib.mmae_set_sm_budget(args.sm_budget)
    # ------------------------------------------------------------------ roofline of the dominant kernel (tcgen05 GEMM): one
    # eager step with CUDA events around every GEMM launch, taken BEFORE the step is captured (a captured graph cannot be
    # profiled per launch, and eager collectives must not be mixed in behind captured ones)
    for _ in range(2):
        stepper._step(resident[0])
    torch.cuda.synchronize()
    peak_tf, peak_gbs, peak_src = peaks()
    # The profiled step runs the four task decoders one after the other on ONE stream: an event pair around a launch measures
    # that launch only when nothing else shares the SMs - with the decoders on their own streams (the timed legs below) every
    # K=256 GEMM is charged for its neighbours' kernels (25088x256x256: 54 TF/s "measured" that way, ~3x its stand-alone rate)
    streams_on = model.decoder_streams
    model.decoder_streams = False
    stepper._step(resident[0])
    torch.cuda.synchronize()
    lib.mmae_profile_gemm(1)
    l0 = lib.mmae_launch_count()
    stepper._step(resident[0])                             # eager: per-launch events cannot be replayed from a graph
    launches_per_step = lib.mmae_launch_count() - l0
    torch.cuda.synchronize()
    lib.mmae_profile_gemm(0)
    model.decoder_streams = streams_on
    fl, ms_g, n_g = ctypes.c_double(), ctypes.c_double(), ctypes.c_int64()
    lib.mmae_profile_gemm_read(ctypes.byref(fl), ctypes.byref(ms_g), ctypes.byref(n_g))
    gemm_tf = fl.value / (ms_g.value * 1e-3) / 1e12 if ms_g.value > 0 else 0.0
    encoder_tc = None
    if rank == 0:
        try:
            buf = ctypes.create_string_buffer(1 << 20)
            n = lib.mmae_profile_gemm_dump(buf, len(buf))
            agg = {}
            for line in buf.raw[:max(n, 0)].decode().splitlines():
                M_, N_, K_, fl_, ms_ = line.split()
                key = (int(M_), int(N_), int(K_), int(fl_) & 3, int(fl_) >> 8)
                a_ = agg.setdefault(key, [0, 0.0])
                a_[0] += 1
                a_[1] += float(ms_)
            if args.gemm_shapes:
                with open(args.gemm_shapes, "w") as fh:
                    fh.write("%7s %6s %6s %3s %5s %5s %9s %8s\n" % ("M", "N", "K", "maj", "split", "count", "ms_total", "TF/s"))
                    for key, (cnt, ms_) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
                        tf = 2.0 * key[0] * key[1] * key[2] * cnt / (ms_ * 1e-3) / 1e12
                        fh.write("%7d %6d %6d %3d %5d %5d %9.3f %8.1f\n" % (key + (cnt, ms_, tf)))
            encoder_tc = encoder_tc_from_table(agg, args.batch * (wl["visible"] + 1), 768 if wl["size"] == "base" else 1024,
                                               peak_tf)
        except Exception as e:  # noqa: BLE001  (diagnostics only: never cost the headline line)
            _note("per-shape GEMM table unavailable: %s" % str(e)[:120])

    mode = "eager"
    if args.graph:
        try:
            stepper.capture(resident[0], warmup=3)
            mode = "cuda-graph (whole step = one graph launch)"
        except Exception as e:  # noqa: BLE001
            stepper.graph = None
            model.external_shares = None
            mode = "eager (graph capture failed: %s)" % str(e).splitlines()[0][:120]

    def train_step(x):
        return stepper(x)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t)
        return ms

    # ------------------------------------------------------------------ leg 1: inputs resident in HBM
    if rank == 0:
        _note("model built, launch mode: %s" % mode)
    for i in range(args.warmup):
        train_step(resident[i % 2])
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = lib.mmae_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        loss, _ = train_step(resident[i % 2])
    e1.record()
    barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    launches = lib.mmae_launch_count() - launches0
    if stepper.graph is not None:
        launches = launches_per_step * args.steps          # a replayed graph re-issues the captured launches
    clocks = sampler.stop() if rank == 0 else None
    final_loss = float(loss)
    if args.dump_outputs:
        # The float atomics of the step (split-K weight gradients, embedding gradients) add in a different order from run
        # to run: rounding-level in one step, but the training steps before the last one compound it.  The dumped step
        # therefore runs the timed path once more, on the last timed batch, from the seeded initial state.
        with torch.no_grad():
            for dst, src in zip(optimizer_state(opt), initial_state):
                dst.copy_(src)
        opt.invalidate_mirror()
        opt.ensure_mirror_fresh()                          # a graph replay does not refresh the bf16 weight twin itself
        loss, grad_norm = train_step(resident[(args.steps - 1) % 2])
        barrier()
        if rank == 0:
            dump_outputs(args.dump_outputs, model, opt, loss, grad_norm)

    if rank == 0:
        _note("leg 1 (HBM-resident inputs): %.3f ms/step" % (ms_total / args.steps))
    # ------------------------------------------------------------------ leg 2: end to end through the public API
    # pinned host inputs -> H2D every step (prefetched on a copy stream, inside the timed region) + loss read back (D2H)
    from multimae_b200.train_step import InputPrefetcher
    feeder = InputPrefetcher(host[0], device)
    h2d_bytes = feeder.bytes_per_batch
    # what the host link of this box delivers for exactly these copies, alone (context for the e2e figure)
    for _ in range(2):
        feeder.submit(host[0])
        feeder.release(feeder.get()[0])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(4):
        feeder.submit(host[i % 2])
        feeder.release(feeder.get()[0])
    torch.cuda.synchronize()
    h2d_gbs = 4 * h2d_bytes / (time.perf_counter() - t0) / 1e9
    if rank == 0:
        _note("H2D of one input batch alone: %.1f MB at %.1f GB/s = %.2f ms" % (h2d_bytes / 1e6, h2d_gbs, h2d_bytes / h2d_gbs / 1e6))

    # The loss of every step is read on the host exactly once, one step late: its D2H copy into a pinned slot is enqueued
    # behind the step, and the host waits for it only after the NEXT step has been launched, so the device never idles
    # on the host round trip (the reference's `loss.item()` right after the step stalls the launch queue every step).
    loss_slots = [torch.zeros(1, dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_events = [torch.cuda.Event() for _ in range(2)]
    def e2e_leg(use_graph):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        feeder.submit(host[0])
        host_losses = []
        for i in range(args.steps):
            slot, cur = feeder.get()
            if i + 1 < args.steps:
                feeder.submit(host[(i + 1) % 2])
            loss, _ = stepper(cur, use_graph=use_graph)
            feeder.release(slot)
            loss_slots[i % 2].copy_(loss.detach().reshape(1), non_blocking=True)      # D2H read of the step's result
            loss_events[i % 2].record()
            if i > 0:
                loss_events[(i - 1) % 2].synchronize()
                host_losses.append(float(loss_slots[(i - 1) % 2]))
        loss_events[(args.steps - 1) % 2].synchronize()
        host_losses.append(float(loss_slots[(args.steps - 1) % 2]))
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    # (The replayed step issues no host -> device copy of its own: a small H2D on the compute stream would queue behind the
    # in-flight 106 MB input copy on the H2D engine and stall the step by the ~2 ms that copy takes - measured.)
    ms_e2e, e2e_mode = e2e_leg(True), ("cuda-graph" if stepper.graph is not None else "eager")

    if rank == 0:
        _note("leg 2 (pinned host inputs, loss read back): %.3f ms/step" % (ms_e2e / args.steps))
    if args.e2e_probe:
        def timed(use_h2d, consume, read_loss, submit_after=False):
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            if use_h2d:
                feeder.submit(host[0])
            for i in range(args.steps):
                cur = resident[i % 2]
                if use_h2d:
                    slot, got = feeder.get()
                    if consume:
                        cur = got
                    if i + 1 < args.steps and not submit_after:
                        feeder.submit(host[(i + 1) % 2])
                loss, _ = train_step(cur)
                if use_h2d:
                    feeder.release(slot)
                    if i + 1 < args.steps and submit_after:
                        feeder.submit(host[(i + 1) % 2])
                if read_loss:
                    loss_slots[i % 2].copy_(loss.detach().reshape(1), non_blocking=True)
                    loss_events[i % 2].record()
                    if i > 0:
                        loss_events[(i - 1) % 2].synchronize()
            b.record()
            barrier()
            return a.elapsed_time(b) / args.steps
        for name, cfg in (("no H2D, no loss read", (False, False, False)), ("no H2D, loss read", (False, False, True)),
                          ("H2D not consumed, loss read", (True, False, True)), ("H2D consumed, no loss read", (True, True, False)),
                          ("H2D consumed, loss read", (True, True, True)),
                          ("H2D consumed, loss read, submit after launch", (True, True, True, True))):
            _note("probe %-46s %.3f ms/step" % (name, timed(*cfg)))
    if world > 1:
        # the captured graph holds NCCL work: release it, drain the device, line the ranks up, then tear the group down
        stepper.graph = None
        torch.cuda.synchronize()
        dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    ms_step = ms_total / args.steps
    value = args.batch * world / (ms_step * 1e-3)
    e2e_value = args.batch * world / (ms_e2e / args.steps * 1e-3)
    out = {
        "metric": wl["metric"], "value": round(value, 1), "unit": "samples/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(ms_step, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": wl["name"] + (" + truncated depth standardisation" if args.standardize_depth else ""),
                   "global_batch": args.batch * world, "per_gpu_batch": args.batch,
                   "parallelism": "dp%d" % world,
                   "l2": "two alternating input batches (212 MB) and a >9 GB per-step activation working set exceed the 126 MB L2",
                   "loss_scaling": "none (bf16)",
                   "sm_budget": args.sm_budget or None,
                   "e2e_pipeline": "H2D of step i+1 prefetched on a copy stream during step i; every step's loss read on "
                                   "the host once, one step late (pinned D2H behind the step)", "final_loss": round(final_loss, 4), "launch_mode": mode},
        "e2e": {"value": round(e2e_value, 1), "unit": "samples/s", "h2d_bytes_per_step": h2d_bytes,
                "d2h_bytes_per_step": 4, "h2d_link_gbs_measured": round(h2d_gbs, 1), "launch_mode": e2e_mode},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"bound": "tensor", "kernel": "gemm_bf16_kernel (tcgen05, all operand-major variants)",
                     "achieved": round(gemm_tf, 1), "peak": peak_tf, "unit": "TFLOP/s",
                     "frac": round(gemm_tf / peak_tf, 4), "traffic": None,
                     "traffic_note": None, "peak_source": peak_src + " (sustained bf16)",
                     "launches_per_step": int(n_g.value), "kernel_ms_per_step": round(ms_g.value, 3),
                     "kernel_share_of_step": round(ms_g.value / ms_step, 3),
                     "how": "CUDA events around every GEMM launch of one eager step with the task decoders serialised on one "
                            "stream (launch-only durations); the timed legs run them on four streams inside one CUDA graph",
                     "step_model_flops_frac": round(value / world * wl["flop"] / (peak_tf * 1e12), 4)},
    }
    if encoder_tc is not None:
        out["encoder_tc"] = encoder_tc
    ev = ncu_evidence() if args.workload == "cfg2" else None
    gemm_ev = (ev or {}).get("dominant_gemm")
    if gemm_ev:          # dram__bytes_read + dram__bytes_write of one launch of the dominant GEMM, from the committed capture
        out["roofline"]["traffic"] = gemm_ev.get("dram_bytes")
        out["roofline"]["traffic_note"] = "%s: %s (ncu --set full, commit %s, profiles/ncu_hot_kernels.json)" % (
            gemm_ev.get("what"), gemm_ev.get("note"), ev.get("commit"))
    else:
        out["roofline"]["traffic_note"] = "no committed ncu capture for this workload's GEMM shapes"
    if world == 1 and args.eager_baseline:
        # free this process's ~10 GB of activations / graph memory pools first: the eager oracle needs room of its own
        _note("GPU legs done (%.1f samples/s); timing torch eager (oracle port) on this GPU" % value)
        out["torch_eager_same_gpu"] = gpu_eager_baseline_bounded(workload=args.workload)
        if out["torch_eager_same_gpu"].get("bf16_autocast"):
            out["torch_eager_same_gpu"]["speedup_vs_bf16_autocast"] = round(value / out["torch_eager_same_gpu"]["bf16_autocast"], 2)
    if world == 1 and args.cpu_baseline:
        _note("timing the CPU baseline sample")
        out["cpu_baseline"] = cpu_baseline_bounded(workload=args.workload)
    _emit(out)
    if world > 1:
        dist.destroy_process_group()


# ----------------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port (oracle/multimae_oracle.py) on the host cores — test infrastructure timed as the baseline
# ----------------------------------------------------------------------------------------------------------------------
def _cpu_steps(batch, steps, warmup, threads=None, workload="cfg2"):
    from oracle import multimae_oracle as O
    wl = WORKLOADS[workload]
    torch.set_num_threads(threads or (os.cpu_count() or 1))
    cfg = O.make_config(size=wl["size"])          # posemb_grid stays 14: tables resized to the input's grid as in get_model
    p = O.init_params(cfg, seed=0)
    train = O.trainable(p)
    for v in train.values():
        v.requires_grad_(True)
    x = O.synthetic_inputs(cfg, batch, wl["image"], seed=0)
    shares, noises, noise_all = O.synthetic_mask_draws(cfg, batch, wl["image"], seed=1)
    m, ids_keep, ids_restore = O.sample_masks(shares, noises, noise_all, wl["visible"])
    tmask = {d.name: mm for d, mm in zip(cfg.in_domains, m)}
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        for v in train.values():
            v.grad = None
        losses, _ = O.step_losses(p, x, cfg, tmask, ids_keep, ids_restore)
        sum(losses.values()).backward()
        O.grad_norm([v.grad for v in train.values()])
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    return times


def _best_thread_count(batch, workload="cfg2"):
    """torch's CPU kernels collapse when a 100+-core host is oversubscribed by this small problem: give the CPU arm
    the thread count at which it is FASTEST (one probe step each), which is the fair baseline."""
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64) if c <= ncpu}) or [ncpu]
    best, best_t = cands[0], float("inf")
    t_begin = time.perf_counter()
    for c in cands:                      # ascending; stop once more threads make it slower, or the probe budget is spent
        t = _cpu_steps(batch, 1, 1, threads=c, workload=workload)[0]
        if t < best_t:
            best, best_t = c, t
        elif t > 1.2 * best_t:
            break
        if time.perf_counter() - t_begin > 40.0:
            break
    return best


def cpu_baseline(sample_steps=2, batch=4, workload="cfg2"):
    threads = _best_thread_count(batch, workload)
    times = _cpu_steps(batch, sample_steps, 1, threads=threads, workload=workload)
    med = statistics.median(times)
    return {"value": round(batch / med, 2), "unit": "samples/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": "%d steps of fwd+4 losses+bwd at bs=%d (same model/inputs shape, fp32, oracle port of the reference "
                      "PyTorch path; no optimizer step; thread count chosen by a probe over 8/16/32/64)" % (sample_steps, batch)}


def _gpu_eager_steps(workload, dtype, steps=5, warmup=2):
    """The oracle port of the reference PyTorch path, eager, on THIS GPU under torch.autocast (fp16 as the reference ships
    it, run_pretraining_multimae.py:500, or bf16): forward + 4 losses + backward at the workload's batch - the "kernel to
    beat" of SURVEY.md section 8(d).  Test infrastructure timed as a baseline, like the CPU arm."""
    from oracle import multimae_oracle as O
    wl = WORKLOADS[workload]
    dev = torch.device("cuda", 0)
    cfg = O.make_config(size=wl["size"])
    p = {k: v.to(dev) for k, v in O.init_params(cfg, seed=0).items()}
    train = O.trainable(p)
    for v in train.values():
        v.requires_grad_(True)
    B = wl["batch"]
    x = {k: v.to(dev) for k, v in O.synthetic_inputs(cfg, B, wl["image"], seed=0).items()}
    shares, noises, noise_all = O.synthetic_mask_draws(cfg, B, wl["image"], seed=1)
    m, ids_keep, ids_restore = O.sample_masks(shares, noises, noise_all, wl["visible"])
    tmask = {d.name: mm.to(dev) for d, mm in zip(cfg.in_domains, m)}
    ids_keep, ids_restore = ids_keep.to(dev), ids_restore.to(dev)
    times = []
    for i in range(warmup + steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for v in train.values():
            v.grad = None
        if dtype is None:
            losses, _ = O.step_losses(p, x, cfg, tmask, ids_keep, ids_restore)
        else:
            with torch.autocast("cuda", dtype=dtype):
                losses, _ = O.step_losses(p, x, cfg, tmask, ids_keep, ids_restore)
        (sum(losses.values()) * (65536.0 if dtype == torch.float16 else 1.0)).backward()
        b.record()
        torch.cuda.synchronize()
        if i >= warmup:
            times.append(a.elapsed_time(b))
    return B / (statistics.median(times) * 1e-3)


def gpu_eager_baseline(workload="cfg2"):
    out = {"unit": "samples/s", "what": "oracle port of the reference PyTorch path, eager on this GPU, fwd+4 losses+bwd at the "
           "workload's batch (no optimizer step), median of 5 steps after 2 warm-ups, CUDA events"}
    for name, dt in (("fp16_autocast", torch.float16), ("bf16_autocast", torch.bfloat16)):
        try:
            out[name] = round(_gpu_eager_steps(workload, dt), 1)
        except Exception as e:  # noqa: BLE001
            out[name] = None
            out[name + "_error"] = str(e).splitlines()[0][:160] if str(e) else type(e).__name__
        torch.cuda.empty_cache()
    return out


def gpu_eager_baseline_bounded(limit_s=150, workload="cfg2"):
    """In a child process (its ~40 GB of eager activations are gone when it exits) with a hard time limit."""
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "gpu-eager", "--workload", workload],
                           capture_output=True, text=True, timeout=limit_s)
        for line in reversed(r.stdout.splitlines()):
            if line.startswith("{"):
                return json.loads(line)
        return {"fp16_autocast": None, "bf16_autocast": None,
                "note": "failed: " + (r.stderr.strip().splitlines() or ["no output"])[-1][:200]}
    except subprocess.TimeoutExpired:
        return {"fp16_autocast": None, "bf16_autocast": None, "note": "exceeded %d s" % limit_s}


def cpu_baseline_bounded(limit_s=150, workload="cfg2"):
    """The CPU sample in a child process with a hard time limit: a slow or oversubscribed host must not cost the GPU line."""
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "cpu-baseline", "--workload", workload],
                           capture_output=True, text=True, timeout=limit_s)
        for line in reversed(r.stdout.splitlines()):
            if line.startswith("{"):
                return json.loads(line)
        note = "CPU sample failed: " + (r.stderr.strip().splitlines() or ["no output"])[-1][:200]
    except subprocess.TimeoutExpired:
        note = "CPU sample exceeded %d s on this host" % limit_s
    return {"value": None, "unit": "samples/s", "cores": 0, "kind": "port", "sample": note}


def run_reference(args, rank, world):
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    # the workload's own batch (cfg2: bs = 128, a few seconds per step on the host cores), so that the arm's config IS the
    # GPU arm's; the thread count is probed at a small batch, the step count is bounded
    batch = wl["batch"] if args.workload == "cfg2" else 2
    threads = _best_thread_count(8 if args.workload == "cfg2" else 2, args.workload)
    steps = min(args.steps, 3)
    times = _cpu_steps(batch, steps, 1, threads=threads, workload=args.workload)
    ms_step = statistics.mean(times) * 1e3
    value = batch / (ms_step * 1e-3)
    base = {"value": round(value, 2), "unit": "samples/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": "%d steps (after 1 warm-up) of fwd+4 losses+bwd+grad-norm at bs=%d on the host cores, fp32, no optimizer "
                      "update (the oracle port of the reference path; bounded step count)" % (steps, batch)}
    _emit({
        "impl": "reference", "metric": wl["metric"], "value": round(value, 2), "unit": "samples/s", "n_gpus": world,
        "steps": steps, "warmup": 1, "ms_per_step": round(ms_step, 1), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["name"], "global_batch": batch, "per_gpu_batch": batch,
                   "note": "CPU arm: oracle port of the reference path (the reference is pure PyTorch and /root/reference "
                           "does not travel to the GPU box); fp32 on the host cores, no optimizer update; with N > 1 it is "
                           "still ONE host process - compare it with the N = 1 line only"},
        "cpu_baseline": base,
        "e2e": {"value": round(value, 2), "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=None, help="per-GPU batch (default: the workload's, 128 for cfg2)")
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS),
                    help="cfg2: MultiMAE-B 224 bs=128 (BASELINE metric, default); cfg4: MultiMAE-L bs=64; cfg5: MultiMAE-B 448x448 bs=32")
    ap.add_argument("--cpu-baseline", type=int, default=1, help="0: skip the bounded CPU sample (development runs only)")
    ap.add_argument("--standardize-depth", type=int, default=0,
                    help="1: truncated depth standardisation (run_pretraining_multimae.py:487-492) inside the step")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "cpu-baseline", "gpu-eager"])
    ap.add_argument("--graph", type=int, default=1, help="1: replay the step as one CUDA graph (data parallel: the bucketed NCCL "
                         "all-reduces are captured in it); 0: eager launches")
    ap.add_argument("--sm-budget", type=int, default=0, help="N>1: SMs the persistent kernels may claim (0 = all; the rest is "
                         "left to NCCL's all-reduce CTAs)")
    ap.add_argument("--eager-baseline", type=int, default=1, help="0: skip the torch-eager-on-this-GPU sample of the oracle port")
    ap.add_argument("--e2e-probe", action="store_true", help="extra timed loops that isolate the H2D / loss-read costs")
    ap.add_argument("--gemm-shapes", default=None, help="write a per-shape GEMM time table of one profiled step here")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, run the timed path once more on the last timed batch from the seeded "
                         "initial state and write what it computed to DIR/<name>.npy (float32; same arguments, same inputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.batch is None:
        args.batch = WORKLOADS[args.workload]["batch"]
    _quiet_stdout()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "cpu-baseline":
        _emit(cpu_baseline(sample_steps=2, batch=4 if args.workload == "cfg2" else 2, workload=args.workload))
        return
    if args.impl == "gpu-eager":
        _emit(gpu_eager_baseline(args.workload))
        return
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    args.warmup = max(args.warmup, 3)
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("launch multi-GPU runs with: python -m torch.distributed.run --nproc-per-node %d bench.py --gpus %d"
                         % (args.gpus, args.gpus))
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
