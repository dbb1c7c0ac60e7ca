#!/usr/bin/env python
"""Benchmark of the WSL4MIS hot path: images/sec of the unet_cct pCE+GatedCRF training step
(train_weakly_supervised_pCE_GatedCRFLoss_2D.py:111-130 replayed on main_seg, SURVEY F7) at 256x256,
batch 64 per GPU, synthetic data, random-init weights.

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W [--scaling strong]
    python bench.py --impl reference ...      # the reference's own modules on the host CPU (staged by oracle/build_ref.py)
    python bench.py ... --dump-outputs DIR    # also write what the last timed step computed as DIR/<name>.npy

Prints ONE JSON line (rank 0).  value = whole-job images/sec with inputs resident in HBM;
e2e = same step driven through the public API from pinned HOST buffers (H2D of the batch and D2H of the loss
inside the timed region).  Extra objects: roofline (dominant kernel) + layers (top launches against their own roofline),
cpu_baseline (the reference on the host cores), gpu_baseline (the reference's modules as stock PyTorch on the same B200),
parity (logit error / label mismatch of every execution mode against the fp32 CUDA-core executor), modes (step time of the
fp16 and fp16x3 modes).
"""
import argparse
import json
import os
import random
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

HW = 256
VARIANT_LABEL = {"uamt": "UAMT (uncertainty-aware mean teacher: Dice+CE + masked consistency, T=8 teacher passes)", "pce": "pCE", "pce_gatedcrf": "pCE+GatedCRF", "pce_ms": "pCE+MumfordShah", "pce_tv": "pCE+TV", "dmpls": "DMPLS (pCE + mixed pseudo-label Dice)",
                 "pce_entropy": "pCE+EntropyMin", "pce_variance": "pCE+ClassVariance"}
CRF_DESC = [{"weight": 1, "xy": 6, "rgb": 0.1}]


def metric_name(args):
    return f"images/sec {args.model} {VARIANT_LABEL.get(args.variant, args.variant)} {HW}x{HW} bs{args.batch}"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=64, help="per-GPU batch (weak scaling) / global batch (--scaling strong)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--model", default="unet_cct", choices=["unet", "unet_cct"])
    ap.add_argument("--variant", default="pce_gatedcrf")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp16", "fp16x3", "fp32"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-kernel-table", action="store_true")
    ap.add_argument("--cpu-sample", type=int, default=8, help="images per CPU-baseline step")
    ap.add_argument("--skip-cpu", action="store_true", help="profiling runs: skip the CPU baseline leg")
    ap.add_argument("--skip-e2e", action="store_true", help="profiling runs: skip the host-buffer leg")
    ap.add_argument("--skip-gpu-baseline", action="store_true", help="skip the stock-PyTorch-on-B200 leg")
    ap.add_argument("--skip-extras", action="store_true", help="skip parity / other-mode timing")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    return args


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tf_burst": d["bf16_tflops"], "tf_sustained": d["bf16_tflops_sustained"], "src": "measured"}
    return {"hbm_gbs": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "src": "fallback"}


def host_cores():
    cores = os.cpu_count() or 1
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:
        pass
    try:  # honour a cgroup CPU quota (oversubscribing a quota-limited container is catastrophically slow)
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            cores = max(1, min(cores, int(float(q) / float(per))))
    except Exception:
        pass
    return min(cores, 64)   # torch CPU ops stop scaling (and start thrashing) far below 128 threads on these sizes


def cpu_model():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def synth(n, seed):
    g = torch.Generator().manual_seed(seed)
    img = torch.rand(n, 1, HW, HW, generator=g)
    lab = torch.full((n, HW, HW), 4, dtype=torch.uint8)
    m = torch.rand(n, HW, HW, generator=g) < 0.03
    lab[m] = torch.randint(0, 4, (int(m.sum()),), generator=g, dtype=torch.uint8)
    return img, lab


DUMP_IMAGES = 8


def dump_outputs(path, step, model, loss):
    """What the last timed step hands its caller, as float32 DIR/<name>.npy: `loss`, `logits_head<i>` (every head's logits,
    N x 4 x H x W, for a fixed, seeded sample of DUMP_IMAGES images of the batch: the whole batch is 64 MB per head at
    batch 64) and `state` (the model's state_dict after the SGD update -- parameters and BatchNorm running statistics --
    flattened in state_dict order).  Call it before the next step: the logits of a captured step live in graph memory."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    out = {"loss": loss.detach().reshape(1)}
    heads = getattr(step, "outputs", None) or []
    if heads:
        pick = torch.randperm(heads[0].shape[0], generator=torch.Generator().manual_seed(0))[:DUMP_IMAGES].sort().values
        for i, h in enumerate(heads):
            out[f"logits_head{i}"] = h[pick.to(h.device)]
    out["state"] = torch.cat([v.detach().reshape(-1).float() for v in model.state_dict().values() if v.is_floating_point()])
    for name, t in out.items():
        np.save(os.path.join(path, name + ".npy"), t.float().cpu().numpy())


# ----------------------------------------------------------------------------------------------
# The reference itself (unmodified modules staged by oracle/build_ref.py): CPU arm and stock-PyTorch-on-B200 arm.
# The only places bench.py touches oracle/.
# ----------------------------------------------------------------------------------------------
_REF = {}


def load_reference():
    """-> dict(UNet, UNet_CCT, losses, CRF) from the staged reference files, or None when nothing is staged"""
    if "mods" not in _REF:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import build_ref
        code = build_ref.extract()
        mods = None
        if code is not None:
            sys.path.insert(0, code)
            import importlib
            unet = importlib.import_module("networks.unet")
            crf = importlib.import_module("utils.gate_crf_loss")
            losses = importlib.import_module("utils.losses")
            mods = {"UNet": unet.UNet, "UNet_CCT": unet.UNet_CCT, "CRF": crf.ModelLossSemsegGatedCRF, "losses": losses, "code": code}
        _REF["mods"] = mods
    return _REF["mods"]


def reference_step_fn(mods, model_name, variant, device, amp=False, channels_last=False, unet_only=False):
    """The step body of train_weakly_supervised_pCE_GatedCRFLoss_2D.py:111-126 (or the pCE / MumfordShah variants) on the reference's
    own modules; unet_cct under a single-head script uses main_seg (SURVEY F7)."""
    torch.manual_seed(2022)
    model = (mods["UNet_CCT"] if model_name == "unet_cct" else mods["UNet"])(in_chns=1, class_num=4).to(device)
    if channels_last:
        model = model.to(memory_format=torch.channels_last)
    model.train()
    opt = torch.optim.SGD(model.parameters(), lr=0.01, momentum=0.9, weight_decay=1e-4)
    ce = torch.nn.CrossEntropyLoss(ignore_index=4)
    crf = mods["CRF"]()
    ms = mods["losses"].MumfordShah_Loss()

    def step(x, lab):
        with torch.autocast(device_type="cuda", dtype=torch.bfloat16, enabled=amp):
            out = model(x.contiguous(memory_format=torch.channels_last) if channels_last else x)
        out = (out[0] if isinstance(out, tuple) else out).float()
        soft = torch.softmax(out, dim=1)
        loss = ce(out, lab.long())
        if not unet_only:
            if variant == "pce_gatedcrf":
                loss = loss + 0.1 * crf(soft, CRF_DESC, 5, x, HW, HW)["loss"]
            elif variant == "pce_ms":
                loss = loss + 1e-6 * ms(x, soft)
        opt.zero_grad()
        loss.backward()
        opt.step()
        return loss

    return step


def cpu_reference_time(args, n_img, steps, warmup):
    """the reference step on the host cores; falls back to the oracle port when the reference files are not staged"""
    cores = host_cores()
    torch.set_num_threads(cores)
    mods = load_reference()
    img, lab = synth(n_img, 2022)
    if mods is not None:
        step = reference_step_fn(mods, args.model, args.variant, torch.device("cpu"))
        kind, what = "reference", "unmodified reference modules (networks/unet.py, utils/gate_crf_loss.py, utils/losses.py staged by oracle/build_ref.py) + torch CrossEntropyLoss / optim.SGD"
        run = lambda: step(img, lab)
    else:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import wsl_oracle as O
        O.CRF_IMPL = "unfold"
        cct = args.model == "unet_cct"
        p = O.synth_params(1, 4, ("main_decoder", "aux_decoder1") if cct else ("decoder",), 2022)
        moms = {}

        def run():
            loss, grads, _ = O.full_step(p, img, lab, args.variant, cct)
            trainable = {k: p[k] for k in grads}
            O.sgd_step(trainable, grads, moms, 0.01)
            p.update(trainable)
        kind, what = "port", "oracle/wsl_oracle.py full_step + sgd_step (reference files not staged on this box)"
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        run()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    t = sum(times) / len(times)
    return {"value": n_img / t, "unit": "images/sec", "cores": cores, "cpu": cpu_model(), "kind": kind,
            "sample": f"{n_img} images of 1x{HW}x{HW} per step, {steps} steps after {warmup} warm-up, torch {torch.__version__} fp32, {what} "
                      f"({args.model}, {args.variant})"}, t


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warm = args.steps, max(0, args.warmup)
    cb, t = cpu_reference_time(args, args.cpu_sample, steps, warm)
    line = {"impl": "reference", "metric": metric_name(args), "value": cb["value"], "unit": "images/sec", "n_gpus": args.gpus,
            "steps": steps, "warmup": warm, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.model} {args.variant} train step, {args.cpu_sample}x1x{HW}x{HW} per step on the host CPU "
                                   f"(bounded sample of the {args.batch}-image step: the unfold GatedCRF needs ~0.8 GB per image)",
                       "note": "the reference is pure PyTorch: its own CPU path is the same modules on CPU tensors"},
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def gpu_reference_baseline(args, dev, img_d, lab_d):
    """The reference's modules as stock PyTorch (ATen / cuDNN) on the same B200: the kernel to beat (SURVEY F1, 8(d))."""
    mods = load_reference()
    if mods is None:
        return {"unavailable": "reference files not staged (oracle/_ref/reference_code.tar missing)"}
    out = {"source": "unmodified reference modules on cuda (oracle/build_ref.py), torch " + torch.__version__, "runs": []}
    saved = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark,
             torch.backends.cudnn.deterministic)
    modes = [("fp32 (scripts' --deterministic 1: cudnn.deterministic, no TF32)", dict(tf32=False, det=True, amp=False, cl=False)),
             ("tf32 + cudnn.benchmark", dict(tf32=True, det=False, amp=False, cl=False)),
             ("amp bf16 + channels_last + cudnn.benchmark", dict(tf32=True, det=False, amp=True, cl=True))]
    try:
        for name, o in modes:
            for unet_only in (False, True):
                torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = o["tf32"]
                torch.backends.cudnn.benchmark, torch.backends.cudnn.deterministic = (not o["det"]), o["det"]
                res = None
                for bs in (args.batch, 32, 16, 8):
                    if bs > args.batch:
                        continue
                    try:
                        torch.cuda.empty_cache()
                        torch.cuda.reset_peak_memory_stats(dev)
                        step = reference_step_fn(mods, args.model, args.variant, dev, o["amp"], o["cl"], unet_only)
                        x, lab = img_d[:bs].contiguous(), lab_d[:bs].contiguous()
                        for _ in range(3):
                            step(x, lab)
                        torch.cuda.synchronize()
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        n = 5
                        e0.record()
                        for _ in range(n):
                            loss = step(x, lab)
                        e1.record()
                        torch.cuda.synchronize()
                        ms = e0.elapsed_time(e1) / n
                        res = {"mode": name, "step": "pCE only (U-Net fwd+bwd+SGD)" if unet_only else f"{args.variant} full step", "batch": bs,
                               "ms_per_step": round(ms, 3), "images_per_sec": round(bs / ms * 1e3, 1),
                               "peak_mem_GiB": round(torch.cuda.max_memory_allocated(dev) / 2 ** 30, 2), "loss": float(loss.detach())}
                        del step
                        break
                    except torch.cuda.OutOfMemoryError:
                        res = None
                        continue
                out["runs"].append(res if res is not None else {"mode": name, "error": "out of memory at every batch size tried"})
    finally:
        (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark,
         torch.backends.cudnn.deterministic) = saved
        torch.cuda.empty_cache()
    full = [r for r in out["runs"] if r and "images_per_sec" in r and r["step"].endswith("full step")]
    if full:
        best = max(full, key=lambda r: r["images_per_sec"])
        out["best_full_step"] = {"mode": best["mode"], "images_per_sec": best["images_per_sec"], "batch": best["batch"]}
    return out


# ----------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out = self.proc.communicate(timeout=5)[0]
        except Exception:
            out = ""
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in out.splitlines():
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        med = sm[len(sm) // 2] if sm else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def parity_report(args, dev):
    """Every execution mode against the fp32 CUDA-core executor (itself pinned to the reference at 1e-5, tests/test_gpu_unet.py) on
    the same weights and an 8 x 1 x 256 x 256 batch, training-mode forward with keep-all dropout masks: max |logit error| as a
    fraction of max |logit| and the fraction of pixels whose argmax differs (north_star: 1e-3 / bit-exact)."""
    from wsl4mis_b200.networks.unet import UNet, UNet_CCT
    n = 8
    img, _ = synth(n, 77)
    x = img.to(dev)
    ft = [16, 32, 64, 128, 256]
    ones = {i: torch.ones(n, HW >> i, HW >> i, ft[i], dtype=torch.uint8, device=dev) for i in range(5)}
    torch.manual_seed(2022)
    base = (UNet_CCT if args.model == "unet_cct" else UNet)(1, 4)
    sd = base.state_dict()
    outs = {}
    for prec in ("fp32", "bf16", "fp16", "fp16x3"):
        m = (UNet_CCT if args.model == "unet_cct" else UNet)(1, 4)
        m.load_state_dict(sd)
        m = m.to(dev).set_precision(prec)
        m.dropout_masks = ones
        if args.model == "unet_cct":
            m.channel_keep = [torch.ones(n, c, dtype=torch.uint8, device=dev) for c in ft]
        m.train()
        with torch.no_grad():
            o = m(x)
        outs[prec] = (o[0] if isinstance(o, tuple) else o).float()
        del m
    ref = outs["fp32"]
    scale = ref.abs().max().item()
    rep = []
    for prec in ("bf16", "fp16", "fp16x3"):
        rep.append({"mode": prec, "logit_err": float((outs[prec] - ref).abs().max().item() / scale),
                    "label_mismatch": float((outs[prec].argmax(1) != ref.argmax(1)).float().mean().item())})
    torch.cuda.empty_cache()
    return {"reference": "fp32 CUDA-core executor (pinned to the reference fixtures at 1e-5)", "batch": f"{n}x1x{HW}x{HW}, train-mode forward, main_seg",
            "tolerance": "north_star: logits within 1e-3 of scale, label maps bit-exact", "modes": rep}


def time_other_modes(args, dev, img_d, lab_d, world):
    """step time of the non-default precision modes (graph mode, device-resident inputs, single process)"""
    from wsl4mis_b200.engine import TrainStep
    from wsl4mis_b200.networks.unet import UNet, UNet_CCT
    out = {}
    for prec in ("bf16", "fp16", "fp16x3"):
        if prec == args.precision:
            continue
        torch.manual_seed(2022)
        m = (UNet_CCT if args.model == "unet_cct" else UNet)(1, 4).to(dev).set_precision(prec)
        st = TrainStep(m, args.variant, graph=True, world_size=1)
        for _ in range(4):
            st(img_d, lab_d)
        torch.cuda.synchronize()
        n = 3 if prec == "fp16x3" else 10
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            st(img_d, lab_d)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        out[prec] = {"ms_per_step": round(ms, 3), "images_per_sec": round(img_d.shape[0] / ms * 1e3, 1)}
        del st, m
        torch.cuda.empty_cache()
    return out


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    from wsl4mis_b200 import _lib
    from wsl4mis_b200.engine import TrainStep
    from wsl4mis_b200.networks.unet import UNet, UNet_CCT

    # weak scaling: --batch images per GPU; strong scaling: --batch images in total (config 4's sweep)
    N = args.batch if args.scaling == "weak" else max(1, args.batch // world)
    torch.manual_seed(2022)
    random.seed(2022)          # dmpls draws its mixing weight from Python's RNG, as the script does
    model = (UNet_CCT if args.model == "unet_cct" else UNet)(1, 4).to(dev).set_precision(args.precision)
    uamt = args.variant == "uamt"
    if uamt:
        # BASELINE config 5 (train_uncertainty_aware_mean_teacher_2D.py:138-197): the per-GPU batch is half labelled (dense labels)
        # and half unlabelled; the teacher is a second, never-updated network (SURVEY F8); main_seg on both sides for unet_cct (F7)
        from wsl4mis_b200.engine import UAMTStep
        torch.manual_seed(2023)
        ema = (UNet_CCT if args.model == "unet_cct" else UNet)(1, 4).to(dev).set_precision(args.precision)
        for q in ema.parameters():
            q.detach_()
        ustep = UAMTStep(model, ema, base_lr=0.01, max_iterations=30000, world_size=world, graph=not args.no_graph)

        class _U:                                    # the TrainStep surface bench.py drives
            # graph_enabled = False: no input_buffers() protocol (UAMTStep copies every batch into its own static buffers);
            # `captured` is what the JSON line reports as cuda_graph
            graph_enabled, captured, launches_per_step, ex = False, ustep.graph_enabled, 0, ustep.ex

            def __call__(self, img, lab):
                h = img.shape[0] // 2
                c0 = _lib.COUNTERS["launch_calls"]
                out = ustep(img[:h], lab[:h], img[h:])
                if ustep.graph_enabled:
                    self.launches_per_step = ustep.launches_per_step      # counted during the eager warm-up steps
                    self.comm_mode = getattr(ustep, "comm_mode", None)
                else:
                    self.launches_per_step = _lib.COUNTERS["launch_calls"] - c0
                return out
        step = _U()
    else:
        step = TrainStep(model, args.variant, base_lr=0.01, max_iterations=30000, graph=not args.no_graph, world_size=world)

    # synthetic batch (SURVEY 8(d)): image ~ U[0,1), ~3 % scribble pixels; different per rank
    img_h, lab_h = synth(N, 2022 + rank)
    if uamt:                                        # --sup_type label: dense labels 0..3
        lab_h = torch.randint(0, 4, lab_h.shape, generator=torch.Generator().manual_seed(99 + rank), dtype=torch.uint8)
    img_h, lab_h = img_h.pin_memory(), lab_h.pin_memory()
    img_d, lab_d = img_h.to(dev), lab_h.to(dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up (>= 3: two eager steps allocate everything, the third captures the graph) ----
    W = max(args.warmup, 3)
    for _ in range(W):
        loss = step(img_d, lab_d)
    barrier()
    first_loss = float(loss.item())

    # ---- timed region 1: device-resident inputs ----
    K = args.steps
    sampler = ClockSampler(local) if rank == 0 else None
    c0 = _lib.COUNTERS["launch_calls"]
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(K):
        loss = step(img_d, lab_d)
    ev1.record()
    barrier()
    ms_dev = ev0.elapsed_time(ev1)
    launches_eager = _lib.COUNTERS["launch_calls"] - c0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, step, model, loss)

    # ---- timed region 2: end to end from pinned host memory, loss read back every step ----
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    copy_stream = torch.cuda.Stream(device=dev)
    main_stream = torch.cuda.current_stream()
    copied = [torch.cuda.Event(), torch.cuda.Event()]
    bufs = [step.input_buffers(0), step.input_buffers(1)] if step.graph_enabled else [(img_d, lab_d), (img_d.clone(), lab_d.clone())]
    bufs[1][0].copy_(img_d)
    bufs[1][1].copy_(lab_d)
    step(*bufs[1])                                   # captures the second graph outside the timed region
    torch.cuda.synchronize()

    def prefetch(i):
        """H2D of one batch from pinned host memory on the copy stream (overlaps the previous step's graph)"""
        with torch.cuda.stream(copy_stream):
            bufs[i][0].copy_(img_h, non_blocking=True)
            bufs[i][1].copy_(lab_h, non_blocking=True)
            copied[i].record(copy_stream)

    loss_h = torch.zeros(2, dtype=torch.float32).pin_memory()
    read_ev = [torch.cuda.Event(), torch.cuda.Event()]
    barrier()
    e0.record()
    n_e2e = 0 if args.skip_e2e else K
    if n_e2e:
        prefetch(0)
    lv = float("nan")
    for k in range(n_e2e):
        cur = k % 2
        main_stream.wait_event(copied[cur])          # this step's inputs have landed
        loss = step(*bufs[cur])
        loss_h[cur:cur + 1].copy_(loss.detach().reshape(1), non_blocking=True)   # D2H of this step's result ...
        read_ev[cur].record()
        if k + 1 < n_e2e:
            if k >= 1:
                copy_stream.wait_event(read_ev[1 - cur])   # step k-1, the last reader of that buffer pair, has finished
            prefetch((k + 1) % 2)                    # next step's H2D runs under this step's graph
        if k >= 1:                                   # ... consumed on the host one step later (software pipelining:
            read_ev[1 - cur].synchronize()           # the launch of step k is never stalled by reading step k-1)
            lv = float(loss_h[1 - cur])
    if n_e2e:
        read_ev[(n_e2e - 1) % 2].synchronize()
        lv = float(loss_h[(n_e2e - 1) % 2])
    e1.record()
    barrier()
    ms_e2e = max(e0.elapsed_time(e1), 1e-6)
    if args.skip_e2e:
        lv = loss.item()
    clocks = sampler.stop() if sampler is not None else None

    t = torch.tensor([ms_dev, ms_e2e], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_dev, ms_e2e = t.tolist()

    # ---- per-kernel table (eager, CUDA events around every C-ABI launch), rank 0, outside the timed regions ----
    table, roof, layers, launches_per_step = None, None, None, None
    peaks = load_peaks()
    if rank == 0 and not args.no_kernel_table and not uamt:
        prof = _lib.Profiler()
        eager = TrainStep(model, args.variant, graph=False, world_size=1)
        eager.ex.multi_stream = False        # serialise: per-kernel event times are only meaningful without overlap
        eager(img_d, lab_d)
        torch.cuda.synchronize()
        _lib.PROFILE = prof
        n_prof = 2
        for _ in range(n_prof):
            eager(img_d, lab_d)
        _lib.PROFILE = None
        agg = prof.table()
        byname = {}
        for (name, meta), (cnt, ms) in agg.items():
            d = byname.setdefault(name, {"launches": 0, "ms": 0.0, "flops": 0.0, "bytes": 0.0})
            d["launches"] += cnt
            d["ms"] += ms
            if meta is not None:
                d["flops"] += meta[2] * cnt
                d["bytes"] += meta[3] * cnt
        detail = sorted(((name, meta[0], meta[1], cnt, ms / cnt, meta[2] / (ms / cnt * 1e-3) / 1e12, meta[3] / (ms / cnt * 1e-3) / 1e9, meta[2], meta[3])
                         for (name, meta), (cnt, ms) in agg.items() if meta is not None), key=lambda r: -r[3] * r[4])
        # the full per-launch table goes to a temporary file: the tree bench.py runs from may be read-only
        fd, detail_path = tempfile.mkstemp(prefix="wsl4mis_kernel_detail_", suffix=".txt")
        with os.fdopen(fd, "w") as f:
            f.write("entry kind layer launches avg_ms TFLOP/s algorithmic_GB/s\n")
            for r in detail:
                f.write(f"{r[0]} {r[1]} {r[2]} {r[3] // n_prof} {r[4]:.4f} {r[5]:.1f} {r[6]:.0f}\n")
        print(f"per-launch kernel table: {detail_path}", file=sys.stderr)
        # top launches, each against the roofline that bounds it (per-kernel event timing: burst tensor peak, measured copy GB/s)
        ridge = peaks["tf_burst"] * 1e12 / (peaks["hbm_gbs"] * 1e9)
        layers = []
        for r in detail[:12]:
            flops, byts = r[7], r[8]
            tensor_bound = byts > 0 and flops / byts > ridge
            frac = (r[5] / peaks["tf_burst"]) if tensor_bound else (r[6] / peaks["hbm_gbs"])
            layers.append({"entry": r[0], "kind": r[1], "layer": r[2], "launches_per_step": r[3] // n_prof, "us": round(r[4] * 1e3, 1),
                           "tflops": round(r[5], 1), "algorithmic_gbs": round(r[6]), "bound": "tensor" if tensor_bound else "hbm",
                           "frac": round(frac, 3)})
        tot = sum(d["ms"] for d in byname.values())
        launches_per_step = sum(d["launches"] for d in byname.values()) // n_prof
        table = {k: {"launches_per_step": v["launches"] // n_prof, "ms_per_step": round(v["ms"] / n_prof, 4),
                     "share": round(v["ms"] / tot, 4),
                     **({"tflops": round(v["flops"] / (v["ms"] * 1e-3) / 1e12, 2)} if v["flops"] else {}),
                     **({"algorithmic_gbs": round(v["bytes"] / (v["ms"] * 1e-3) / 1e9)} if v["bytes"] and not v["flops"] else {})}
                 for k, v in sorted(byname.items(), key=lambda kv: -kv[1]["ms"])}
        top = max(byname.items(), key=lambda kv: kv[1]["ms"])
        name, v = top
        traffic = None
        for tp in ("r2_traffic.json", "r1_traffic.json"):
            tpath = os.path.join(ROOT, "profiles", tp)
            if os.path.exists(tpath):
                tj = json.load(open(tpath))
                if tj.get("kernel") == name:
                    traffic = {"dram_MB_per_launch": round(tj["dram_bytes_per_launch_MB"], 1), "source": tj["source"]}
                    break
        if v["flops"] > 0:
            ach = v["flops"] / (v["ms"] * 1e-3) / 1e12
            roof = {"kernel": name, "bound": "tensor", "achieved": round(ach, 2), "peak": peaks["tf_burst"], "unit": "TFLOP/s",
                    "frac": round(ach / peaks["tf_burst"], 4), "frac_of_sustained": round(ach / peaks["tf_sustained"], 4), "traffic": traffic,
                    "algorithmic_MB_per_launch": round(v["bytes"] / v["launches"] / 1e6, 1),
                    "peak_source": peaks["src"] + " bf16 burst (kernels timed one by one with CUDA events; the step is not power-limited)",
                    "avg_launch_ms": round(v["ms"] / v["launches"], 4), "algorithmic_flops_per_launch": v["flops"] / v["launches"]}
        else:
            ach = v["bytes"] / (v["ms"] * 1e-3) / 1e9 if v["bytes"] else 0.0
            roof = {"kernel": name, "bound": "hbm", "achieved": round(ach, 1), "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": round(ach / peaks["hbm_gbs"], 4), "traffic": traffic, "peak_source": peaks["src"],
                    "avg_launch_ms": round(v["ms"] / v["launches"], 4), "algorithmic_MB_per_launch": round(v["bytes"] / v["launches"] / 1e6, 1)}

    lps, graph_on = step.launches_per_step, getattr(step, "captured", step.graph_enabled)   # launches per step counted at capture time
    parity = modes = gpu_base = None
    if rank == 0 and world == 1 and not args.skip_extras and not uamt:
        parity = parity_report(args, dev)
        modes = time_other_modes(args, dev, img_d, lab_d, world)
    if rank == 0 and world == 1 and not args.skip_gpu_baseline and not uamt:
        del step
        torch.cuda.empty_cache()
        gpu_base = gpu_reference_baseline(args, dev, img_d, lab_d)

    if rank == 0:
        cb = None if (args.skip_cpu or uamt or world > 1) else cpu_reference_time(args, args.cpu_sample, 3, 1)[0]   # rank 0 at N = 1 only
        imgs = N * world * K
        line = {
            "metric": metric_name(args), "value": imgs / (ms_dev * 1e-3), "unit": "images/sec", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": {"bf16": "bf16", "fp16": "f16", "fp16x3": "f32 (fp16 hi/lo split tensor-core products)", "fp32": "f32"}[args.precision],
            "data": "synthetic",
            "config": {"workload": f"{args.model} {args.variant} train step (fwd+loss+bwd+SGD), {N}x1x{HW}x{HW} per GPU, "
                                   f"loss on main_seg (SURVEY F7)", "global_batch": N * world, "parallelism": f"dp{world}",
                       "precision": args.precision, "cuda_graph": bool(graph_on),
                       "comm": getattr(step, "comm_mode", None) if world > 1 else None,
                       "bn": "per-rank batch statistics (stock DDP semantics)",
                       "l2": "per-step working set (~6 GB of activations) >> 126 MB L2; no explicit flush needed"},
            "e2e": {"value": imgs / (ms_e2e * 1e-3), "unit": "images/sec", "ms_per_step": ms_e2e / K,
                    "h2d_bytes_per_step": int(img_h.numel() * 4 + lab_h.numel()), "d2h_bytes_per_step": 4},
            "gpu_launches": (lps * K) if graph_on else launches_eager,
            "gpu_launches_per_step": lps,
            "clocks": clocks, "roofline": roof, "layers": layers, "cpu_baseline": cb, "gpu_baseline": gpu_base, "parity": parity, "modes": modes,
            "kernels": table, "loss_first": first_loss, "loss_last": float(lv),
        }
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
