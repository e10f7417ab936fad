#!/usr/bin/env python
"""bench.py -- headline benchmark of the fake-quant hot path on B200.

Workload (BASELINE.json configs[1]): the quantize->dequantize work of ONE ResNet-50 QAT forward at
batch 256, 8w8a: the 55 activation quantizer sites (per-tensor 8-bit, fused QDQ + MinMax-observer
statistics kernel -- the kernel the 70 %-of-HBM-roofline target is quoted on) and the 54 weight
quantizer sites (per-channel symmetric 8-bit).  A "step" is one pass over all 109 sites on
synthetic tensors of exactly those shapes.  metric = fake-quant forward Gelem/s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

N > 1 is launched by torchrun (one rank per GPU); the path has no exchange step, so ranks are
independent replicas (weak scaling) and only the timing barrier uses NCCL.

--dump-outputs DIR writes what rank 0's last timed step computed as DIR/<name>.npy (float32), so that
two builds run with the same arguments (hence the same seeded inputs) can be compared output for output.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "fake-quant fwd Gelem/s"
UNIT = "Gelem/s"
WORKLOAD = ("resnet50_qat_fwd_8w8a_bs256 (BASELINE configs[1]): 55 activation sites per-tensor 8-bit "
            "fused QDQ+MinMax stats, 54 weight sites per-channel symmetric 8-bit")


# ------------------------------------------------------------------------------------------------
# ResNet-50 quantizer sites (torchvision v1.5 layout: stride on the 3x3), SURVEY.md section 3.2
def r50_activation_sites(bs):
    """Input tensor of every QConv2d (53) + QAdaptiveAvgPool2d + QLinear = 55 sites; (shape, post_relu)."""
    sites = [((bs, 3, 224, 224), False)]
    inplanes, hw = 64, 56
    for planes, blocks, stride in [(64, 3, 1), (128, 4, 2), (256, 6, 2), (512, 3, 2)]:
        for b in range(blocks):
            s = stride if b == 0 else 1
            sites.append(((bs, inplanes, hw, hw), True))            # conv1 1x1
            sites.append(((bs, planes, hw, hw), True))              # conv2 3x3 (stride s)
            hw2 = hw // s
            sites.append(((bs, planes, hw2, hw2), True))            # conv3 1x1
            if b == 0:
                sites.append(((bs, inplanes, hw, hw), True))        # downsample 1x1
            inplanes, hw = planes * 4, hw2
    sites.append(((bs, 2048, 7, 7), True))                          # avgpool input
    sites.append(((bs, 2048), False))                               # fc input
    return sites


def r50_weight_sites():
    ws = [(64, 3, 7, 7)]
    inplanes = 64
    for planes, blocks in [(64, 3), (128, 4), (256, 6), (512, 3)]:
        for b in range(blocks):
            ws += [(planes, inplanes, 1, 1), (planes, planes, 3, 3), (planes * 4, planes, 1, 1)]
            if b == 0:
                ws.append((planes * 4, inplanes, 1, 1))
            inplanes = planes * 4
    ws.append((1000, 2048))
    return ws


def numel(shape):
    n = 1
    for d in shape:
        n *= d
    return n


DUMP_SAMPLE = 1 << 16  # values written per site: 109 sites stay below 30 MB (a step's outputs are 11 GB)


def dump_outputs(out_dir, acts, weights, mm_states):
    """Write what a step hands its caller: every site's QDQ output (act_qdq_NN / weight_qdq_NN, in site order;
    the whole tensor when it has at most DUMP_SAMPLE elements, else the values at DUMP_SAMPLE positions drawn from
    a fixed seed, sorted) and the (min, max) of the 55 fused MinMax observers (act_minmax, [55, 2])."""
    import numpy as np

    from sparsebit_b200 import ops

    os.makedirs(out_dir, exist_ok=True)
    g = torch.Generator().manual_seed(0)

    def sample(t):
        flat = t.reshape(-1)
        if flat.numel() <= DUMP_SAMPLE:
            return flat
        return flat[torch.randint(flat.numel(), (DUMP_SAMPLE,), generator=g).sort().values.to(flat.device)]

    for prefix, sites in (("act_qdq", acts), ("weight_qdq", weights)):
        for i, site in enumerate(sites):
            np.save(os.path.join(out_dir, f"{prefix}_{i:02d}.npy"), sample(site[1]).cpu().numpy())
    mn, mx = ops.minmax_read(mm_states)
    np.save(os.path.join(out_dir, "act_minmax.npy"), torch.stack([mn, mx], dim=1).cpu().numpy())


# ------------------------------------------------------------------------------------------------
def cpu_reference_pass(acts, weights):
    """One pass of the reference's CPU op chain (oracle/torch_port.py) over a sample of the workload."""
    from oracle import torch_port

    for x, s, z in acts:
        torch_port.ort_fake_quant_cpu(x, s, z, 0, 255)
        torch_port.minmax_cpu(x)
    for w, s, z in weights:
        torch_port.ort_fake_quant_cpu(w, s, z, -128, 127)


def build_cpu_sample(sample_bs):
    g = torch.Generator().manual_seed(0)
    acts, weights = [], []
    for shape, relu in r50_activation_sites(sample_bs):
        x = torch.randn(shape, generator=g)
        if relu:
            x = torch.relu(x)
        s = (x.max() - x.min().clamp(max=0)) / 255.0
        acts.append((x, s.reshape(1), torch.round(-x.min().clamp(max=0) / s).reshape(1)))
    for shape in r50_weight_sites():
        w = torch.randn(shape, generator=g) * (2.0 / numel(shape[1:])) ** 0.5
        amax = w.reshape(shape[0], -1).abs().max(dim=1).values
        s = (amax * 2 / 255.0).clamp(min=1e-6).reshape([-1] + [1] * (len(shape) - 1))
        weights.append((w, s, torch.zeros_like(s)))
    elems = sum(x.numel() for x, _, _ in acts) + sum(w.numel() for w, _, _ in weights)
    return acts, weights, elems


def bind_to_gpu_numa(local):
    """Pin this rank's threads (and, by first touch, its pinned host buffers) to the NUMA node its GPU hangs off.
    Round 1's end-to-end numbers scaled non-monotonically (10.4 / 19.6 / 17.4 / 30.1 Gelem/s at 1 / 2 / 4 / 8 GPUs)
    with unbound ranks copying across sockets.  Returns a small report for the JSON line."""
    info = {"numa_node": None, "cpus": None}
    try:
        import pynvml

        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(local)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:  # nvml prints an 8-digit PCI domain, sysfs uses 4
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return info
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            info = {"numa_node": node, "cpus": len(cpus)}
    except Exception as e:  # binding is an optimisation; never fail the benchmark over it
        info["error"] = repr(e)[:120]
    return info


def timed_cpu(fn, budget_s):
    """(seconds per call, calls) of fn on the host, at least one call, about budget_s in total."""
    fn()
    n, t0 = 0, time.perf_counter()
    while True:
        fn()
        n += 1
        dt = time.perf_counter() - t0
        if dt >= budget_s or n >= 50:
            return dt / n, n



# ------------------------------------------------------------------------------------------------
# BASELINE configs[3]: ResNet-50 unstructured L1 sparser mask-apply + 4w4a fake-quant forward, bs 256
def block_sparse_4w4a(lib, dev, acts, weights, peak, steps):
    """One step = `w * mask` + 4-bit per-channel weight QDQ of all 54 weights in ONE multi-tensor launch
    (sb200_qdq_multi_run, 9 B/elem) + the 55 activation sites as 4-bit per-tensor QDQ (8 B/elem).  The masks come
    from the L1 sparser path (radix-select threshold + sb200_mask_gt, ratio 0.5), timed separately."""
    from sparsebit_b200 import _lib, ops

    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    t0, t1 = ev(), ev()
    t0.record()
    masks = []
    for w in weights:
        flat = w[0].reshape(-1)
        k = min(int(flat.numel() * 0.5), flat.numel() - 1)
        masks.append(ops.mask_gt(w[0], ops.kth_value(flat, k, key_mode=1)))
    t1.record()
    torch.cuda.synchronize()
    mask_ms = t0.elapsed_time(t1)
    items = []
    for (w, out, _, _), m in zip(weights, masks):
        amax = (w * m).reshape(w.shape[0], -1).abs().max(dim=1).values
        s4 = (amax * 2 / 15.0).clamp(min=1e-6).contiguous()
        items.append(dict(x=w, mask=m, scale=s4, zero_point=torch.zeros_like(s4), qmin=-8, qmax=7, out=out))
    plan = ops.QdqMulti(items)
    a4 = []
    for a in acts:  # affine 4-bit: scale from the site's range
        mn, mx = a[0].min().clamp(max=0), a[0].max().clamp(min=0)
        s = ((mx - mn) / 15.0).clamp(min=1e-6).reshape(1)
        a4.append((s, torch.round(-mn / s).reshape(1)))
    stream = torch.cuda.current_stream(dev).cuda_stream

    def act_pass(st):
        rc = 0
        for a, (s, z) in zip(acts, a4):
            rc |= lib.sb200_qdq_pertensor_fwd(a[0].data_ptr(), s.data_ptr(), z.data_ptr(), a[1].data_ptr(), a[0].numel(), 0, 15, 0, st)
        if rc:
            _lib.check(rc, "qdq 4-bit")

    def weights_separately(st):
        rc = 0
        for it in items:
            w = it["x"]
            rc |= lib.sb200_mask_apply_qdq_perchannel(w.data_ptr(), it["mask"].data_ptr(), it["scale"].data_ptr(), it["zero_point"].data_ptr(),
                                                      it["out"].data_ptr(), 1, w.shape[0], w.numel() // w.shape[0], -8, 7, 0, st)
        if rc:
            _lib.check(rc, "mask_apply_qdq")

    def timed(fn, reps):
        fn()
        a, b = ev(), ev()
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    launches0 = _lib.launch_count()
    plan.run()
    assert _lib.launch_count() - launches0 == 1
    ref_out = [it["out"].clone() for it in items[:3]]
    weights_separately(stream)
    torch.cuda.synchronize()
    assert all(torch.equal(r, it["out"]) for r, it in zip(ref_out, items[:3])), "multi-tensor launch != per-tensor fused kernels"
    reps = max(3, min(steps, 20))
    multi_ms = timed(plan.run, reps)
    sep_ms = timed(lambda: weights_separately(stream), reps)
    step_ms = timed(lambda: (plan.run(), act_pass(stream)), reps)
    w_elems = sum(it["x"].numel() for it in items)
    a_elems = sum(a[0].numel() for a in acts)
    wb = w_elems * 9.0
    return {"workload": "resnet50 L1-unstructured (ratio 0.5) mask-apply + 4w4a fake-quant forward, bs 256 (BASELINE configs[3])",
            "value": (w_elems + a_elems) / (step_ms * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": step_ms,
            "launches_per_step": 1 + len(acts),
            "weights_one_launch": {"us": multi_ms * 1e3, "GB/s": wb / (multi_ms * 1e-3) / 1e9, "frac": wb / (multi_ms * 1e-3) / 1e9 / peak,
                                   "algorithmic_bytes": wb, "kernel": "sb200::qdq_multi_kernel (54 tensors, 27 560 rows)"},
            "weights_54_launches": {"us": sep_ms * 1e3, "GB/s": wb / (sep_ms * 1e-3) / 1e9, "frac": wb / (sep_ms * 1e-3) / 1e9 / peak},
            "multi_tensor_speedup": sep_ms / multi_ms,
            "mask_generation_ms": mask_ms, "mask_kernels": "sb200_select_* (3-pass radix select, key |w|) + sb200_mask_gt per tensor",
            "parity": "multi-tensor outputs bit-identical to sb200_mask_apply_qdq_perchannel on the first 3 tensors"}


# ------------------------------------------------------------------------------------------------
# BASELINE configs[2]: DeiT-base PTQ observer calibration, 1024-sample set sharded 128 samples / GPU
DEIT_BLOCK_SITES = [(197, 768), (197, 768), (197, 3072), (12, 197, 197)]  # qkv in, fc1 in, fc2 in, attention probabilities


def block_calibration(dev, world, rank, peak, blocks=12, shard=128):
    """Every rank feeds its shard (seed 1000 + rank) into one quantizer per site and all quantizers finish in ONE
    lockstep sweep (sparsebit_b200.distributed.drive_all): statistics of the whole model cross the ranks in one
    packed MAX + one packed SUM all-reduce per round.  Timed with the all-reduces inside, max over ranks."""
    import torch.distributed as dist

    from sparsebit_b200 import config as sbcfg
    from sparsebit_b200 import distributed as sbdist
    from sparsebit_b200.quantization import build_quantizer
    from sparsebit_b200.quantization.common import Backend

    def shard_data(r, nblocks):
        g = torch.Generator(device=dev).manual_seed(1000 + r)
        out = []
        for _ in range(nblocks):
            for shp in DEIT_BLOCK_SITES:
                x = torch.randn((shard,) + shp, device=dev, generator=g)
                if len(shp) == 3:
                    x = torch.softmax(x, dim=-1)  # attention probabilities in [0, 1]
                out.append(x)
        return out

    def make_quantizers(n, observer):
        qs = []
        for i in range(n):
            cfg = sbcfg.quantizer_config("per-tensor-affine" if i % 4 == 3 else "per-tensor-symmetric", 8, "feature", observer, layout="NLC")
            q = build_quantizer(cfg)
            q.set_backend(Backend.VIRTUAL)
            qs.append(q)
        return qs

    if world > 1:
        sbdist.enable()
    data = shard_data(rank, blocks)
    elems = sum(x.numel() for x in data)
    passes = {"minmax": 1, "mse": 2, "percentile": 3}  # reads of the shard: running min/max (+ sweep | 3 radix passes)
    res = {"workload": f"DeiT-base activation sites x{blocks} blocks, {shard} samples per GPU (BASELINE configs[2]), {len(data)} quantizers, "
                       f"{elems} elems per GPU", "world": world, "timing": "second of two sweeps (the first warms NCCL connections and the allocator)",
           "observers": {}}
    check = {}
    for observer in ("minmax", "mse", "percentile"):
        # one untimed warm-up sweep (the first NCCL collective of a given size pays ~30 ms of connection set-up; caching
        # allocator growth), then the timed one on fresh quantizers
        for timed in (False, True):
            qs = make_quantizers(len(data), observer)
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            sbdist.collectives(reset=True)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record()
            for q, x in zip(qs, data):
                q.update_observer(x, alias_ok=True)
            sbdist.drive_all([q.calc_qparams_steps() for q in qs])
            e1.record()
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
        tt = torch.tensor([e0.elapsed_time(e1), wall * 1e3], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt[0])
        coll = sbdist.collectives(reset=True)
        res["observers"][observer] = {
            "ms": ms, "wall_ms": float(tt[1]), "Gelem/s": world * elems / (ms * 1e-3) / 1e9, "collectives": coll,
            "hbm_frac_per_gpu": elems * 4.0 * passes[observer] / (ms * 1e-3) / 1e9 / peak, "data_passes": passes[observer]}
        check[observer] = [(q.scale.reshape(-1).clone(), q.zero_point.reshape(-1).clone()) for q in qs[:4]]
    # bit-exact check: rank 0 rebuilds EVERY shard of the first block and calibrates the whole set alone
    if world > 1:
        sbdist.disable()
    if rank == 0:
        whole = [torch.cat(parts, dim=0) for parts in zip(*[shard_data(r, 1) for r in range(world)])]
        ok = True
        for observer in ("minmax", "mse", "percentile"):
            qs = make_quantizers(4, observer)
            for q, x in zip(qs, whole):
                q.update_observer(x, alias_ok=True)
                q.calc_qparams()
            ok &= all(torch.equal(q.scale.reshape(-1), c[0]) and torch.equal(q.zero_point.reshape(-1), c[1])
                      for q, c in zip(qs, check[observer]))
        res["bit_exact_vs_rank0_whole_set"] = bool(ok)
        del whole
    if world > 1:
        dist.barrier()  # the other ranks wait for rank 0's whole-set check before anything is torn down
    res["collective"] = ("one packed all_reduce(MAX) over order-preserving min/max keys + one packed all_reduce(SUM, fp64) per round "
                         "over NCCL" if world > 1 else "single GPU: no collective")
    del data
    torch.cuda.empty_cache()
    return res


# ------------------------------------------------------------------------------------------------
# BASELINE configs[0]: ResNet-18 PTQ 8w8a MinMax (examples/post_training_quantization/imagenet1k basecase)
def _resnet18_ptq_cpu_port(model, batches):
    """The reference's PTQ pipeline as it runs on the CPU (CalibrationRunner + MinMax observers + quantized forward),
    restated with the torch op chains of oracle/torch_port.py: per-layer activation cache -> cat -> min/max ->
    qparams (tools/calibration.py:100-135, observers/base.py:28,63-79), then a forward with QDQ'd inputs / weights."""
    from oracle import torch_port as tp

    layers = [m for m in model.modules() if isinstance(m, (torch.nn.Conv2d, torch.nn.Linear))]
    cache = {id(m): [] for m in layers}
    hooks = [m.register_forward_pre_hook(lambda mod, args: cache[id(mod)].append(args[0].detach())) for m in layers]
    with torch.no_grad():
        for x in batches:
            model(x)
    for h in hooks:
        h.remove()
    qp = {}
    for m in layers:
        mn, mx = tp.minmax_observer_cpu(cache[id(m)])
        a = tp.calc_qparams_with_minmax_cpu(mn, mx, 0, 255, False)
        w = m.weight.detach()
        rows = w.reshape(w.shape[0], -1)
        ws, wz = tp.calc_qparams_with_minmax_cpu(rows.min(dim=1).values, rows.max(dim=1).values, -128, 127, True)
        shape = [-1] + [1] * (w.dim() - 1)
        qp[id(m)] = (a, (ws.reshape(shape), wz.reshape(shape)))
    saved = {id(m): m.weight.data for m in layers}
    hooks = []
    for m in layers:
        (s, z), (ws, wz) = qp[id(m)]
        m.weight.data = tp.ort_fake_quant_cpu(saved[id(m)], ws, wz, -128, 127)
        hooks.append(m.register_forward_pre_hook(lambda mod, args, s=s, z=z: (tp.ort_fake_quant_cpu(args[0], s, z, 0, 255),)))
    with torch.no_grad():
        y = model(batches[0])
    for h in hooks:
        h.remove()
    for m in layers:
        m.weight.data = saved[id(m)]
    first = layers[0]
    return y, qp[id(first)][0]


def block_resnet18_ptq(dev, n_batches=4, bs=16):
    """ResNet-18 (torchvision architecture, random weights), 8w8a MinMax PTQ on a synthetic 224x224 calibration set:
    ours = host images -> GPU -> streaming CalibrationRunner -> qparams -> quantized forward -> logits back on the host;
    reference arm = the same pipeline restated on the CPU (port)."""
    import torchvision

    from sparsebit_b200 import config as sbcfg
    from sparsebit_b200.quantization.modules import QConv2d, QLinear
    from sparsebit_b200.quantization.tools import CalibrationRunner

    torch.manual_seed(0)
    net = torchvision.models.resnet18(weights=None).eval()
    batches = [torch.randn(bs, 3, 224, 224) for _ in range(n_batches)]
    import copy

    cpu_net = copy.deepcopy(net)
    t0 = time.perf_counter()
    y_cpu, (s_cpu, z_cpu) = _resnet18_ptq_cpu_port(cpu_net, batches)
    cpu_s = time.perf_counter() - t0

    def wrap(module):
        for name, child in list(module.named_children()):
            if isinstance(child, torch.nn.Conv2d):
                setattr(module, name, QConv2d(child).build_quantizer(sbcfg.quantizer_config("per-tensor-affine", 8, "feature"),
                                                                     sbcfg.quantizer_config("per-channel-symmetric", 8, "weight")))
            elif isinstance(child, torch.nn.Linear):
                setattr(module, name, QLinear(child).build_quantizer(sbcfg.quantizer_config("per-tensor-affine", 8, "feature"),
                                                                     sbcfg.quantizer_config("per-channel-symmetric", 8, "weight")))
            else:
                wrap(child)

    old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        qnet = copy.deepcopy(net)
        wrap(qnet)
        qnet = qnet.to(dev)
        pinned = [b.pin_memory() for b in batches]

        def pipeline():
            runner = CalibrationRunner(qnet, streaming=True, record_inputs=False)
            runner.prepare_calibration()
            with torch.no_grad():
                for b in pinned:
                    qnet(b.to(dev, non_blocking=True))
            runner.layerwise_calibration()
            for m in qnet.modules():
                if hasattr(m, "set_quant") and hasattr(m, "input_quantizer"):
                    m.set_quant(w_quant=True, a_quant=True)
            with torch.no_grad():
                y = qnet(pinned[0].to(dev, non_blocking=True)).cpu()
            for m in qnet.modules():
                if hasattr(m, "set_quant") and hasattr(m, "input_quantizer"):
                    m.set_quant(False, False)
            return y

        pipeline()  # warm-up (cuDNN autotune, lazy CUDA init)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        y_gpu = pipeline()
        torch.cuda.synchronize()
        gpu_s = time.perf_counter() - t0
        q0 = qnet.conv1.input_quantizer
        same_first = bool(torch.equal(q0.scale.reshape(-1).cpu(), s_cpu.reshape(-1)) and torch.equal(q0.zero_point.reshape(-1).cpu(), z_cpu.reshape(-1)))
        agree = float((y_gpu.argmax(dim=1) == y_cpu.argmax(dim=1)).float().mean())
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
    imgs = n_batches * bs
    return {"workload": f"ResNet-18 PTQ 8w8a MinMax, {imgs} synthetic 224x224 calibration images + one quantized batch (BASELINE configs[0])",
            "ours_s": gpu_s, "ours_images_per_s": imgs / gpu_s, "cpu_port_s": cpu_s, "cpu_port_images_per_s": imgs / cpu_s,
            "cpu_threads": torch.get_num_threads(), "speedup": cpu_s / gpu_s, "first_layer_qparams_bit_identical": same_first,
            "top1_agreement_with_cpu_port": agree,
            "ours_includes": "H2D of the images from pinned memory, calibration forwards with streaming observers, calc_qparams, quantized forward, D2H of the logits"}


# ------------------------------------------------------------------------------------------------
def block_cpu_baselines(threads):
    """BASELINE.md section 3.1: the reference's CPU paths of the observers / sparser / mask-apply timed on this box's
    host cores (torch op chains of oracle/torch_port.py, pinned to the reference's outputs), next to OUR kernels on
    the same tensors; bounded samples."""
    from oracle import torch_port as tp
    from sparsebit_b200 import config as sbcfg
    from sparsebit_b200 import ops
    from sparsebit_b200.quantization import build_quantizer
    from sparsebit_b200.quantization.common import Backend

    torch.set_num_threads(threads)
    dev = torch.device("cuda", torch.cuda.current_device())
    g = torch.Generator().manual_seed(3)
    x = torch.randn(16, 197, 768, generator=g)  # 2.4 M elems: a DeiT-base site at 16 samples
    w = torch.randn(512, 512, 3, 3, generator=g) * 0.02  # the largest ResNet-50 conv weight
    xd, wd = x.to(dev), w.to(dev)
    out = {"threads": threads, "sample": "observers: [16,197,768] fp32 (2.42 M elems); sparser: [512,512,3,3] (2.36 M elems)"}

    def ours_observer(kind):
        q = build_quantizer(sbcfg.quantizer_config("per-tensor-symmetric", 8, "feature", kind, layout="NLC"))
        q.set_backend(Backend.VIRTUAL)

        def run():
            q.update_observer(xd, alias_ok=True)
            q.calc_qparams()
            torch.cuda.synchronize()

        return run

    mask_dev = ops.mask_gt(wd, ops.kth_value(wd.reshape(-1), wd.numel() // 2, key_mode=1))
    mask_cpu = mask_dev.cpu()
    legs = {
        "minmax_calc_qparams": (lambda: tp.minmax_observer_cpu([x]), ours_observer("minmax")),
        "mse_calc_qparams": (lambda: tp.mse_observer_cpu([x], -128, 127, True), ours_observer("mse")),
        "percentile_calc_qparams": (lambda: tp.percentile_observer_cpu([x], 1e-3), ours_observer("percentile")),
        "kl_calc_qparams": (lambda: tp.kl_observer_cpu([x], 8), ours_observer("kl_histogram")),
        "l1norm_calc_mask": (lambda: tp.l1_unstructured_mask_cpu(w, 0.5),
                             lambda: (ops.mask_gt(wd, ops.kth_value(wd.reshape(-1), wd.numel() // 2, key_mode=1)), torch.cuda.synchronize())),
        "mask_apply": (lambda: tp.mask_apply_cpu(w, mask_cpu), lambda: (ops.mask_apply(wd, mask_dev), torch.cuda.synchronize())),
    }
    for name, (cpu_fn, gpu_fn) in legs.items():
        elems = w.numel() if name in ("l1norm_calc_mask", "mask_apply") else x.numel()
        cs, cn = timed_cpu(cpu_fn, 1.0)
        gs, gn = timed_cpu(gpu_fn, 0.3)
        out[name] = {"cpu_ms": cs * 1e3, "cpu_Melem/s": elems / cs / 1e6, "ours_ms": gs * 1e3, "ours_Melem/s": elems / gs / 1e6,
                     "speedup": cs / gs, "cpu_calls": cn}
    out["note"] = "ours = wall time through the plugin API incl. Python, launches and the final synchronize (device-resident input)"
    return out


def host_threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def pick_cpu_setup(budget_s):
    """Choose the thread count (all usable host threads, or fewer if that is faster -- oversubscribed
    elementwise ATen ops collapse on some hosts) and the sample batch size so that one pass of the
    reference's CPU op chain takes about `budget_s` seconds."""
    probe_acts, probe_w, probe_elems = build_cpu_sample(1)
    best = None
    n = host_threads()
    for threads in sorted({n, min(n, 64), min(n, 32), min(n, 16), min(n, 8)}, reverse=True):
        torch.set_num_threads(threads)
        cpu_reference_pass(probe_acts, probe_w)
        t0 = time.perf_counter()
        cpu_reference_pass(probe_acts, probe_w)
        dt = time.perf_counter() - t0
        if best is None or dt < best[1]:
            best = (threads, dt)
    threads, dt = best
    torch.set_num_threads(threads)
    rate = probe_elems / dt
    per_image = 10_764_800
    bs = int(max(1, min(32, (rate * budget_s - 25_502_912) // per_image)))
    return threads, bs


def time_cpu_baseline(reps, warmup, budget_s=1.0):
    threads, sample_bs = pick_cpu_setup(budget_s)
    acts, weights, elems = build_cpu_sample(sample_bs)
    for _ in range(warmup):
        cpu_reference_pass(acts, weights)
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        cpu_reference_pass(acts, weights)
        times.append(time.perf_counter() - t0)
    return elems, times, threads, sample_bs


def run_reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path (torch op chain of
    quant_tensor.py:181-184 + min/max, all usable host threads) on a bounded sample of the same
    workload; rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    os.environ.pop("OMP_NUM_THREADS", None)  # torchrun pins it to 1
    elems, times, threads, sample_bs = time_cpu_baseline(args.steps, args.warmup, budget_s=1.5)
    total = sum(times)
    value = elems * len(times) / total / 1e9
    sample = (f"all 109 sites at batch {sample_bs} instead of 256 ({elems} elems per step), torch CPU op chain of "
              "quant_tensor.py:181-184 + min/max (oracle/torch_port.py)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": len(times),
        "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "global_batch": 256 * args.gpus, "sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.path = gpu_index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "100"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return None
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for ln in open(self.path):
                f = [p.strip() for p in ln.split(",")]
                if len(f) < 9:
                    continue
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if not sm:
            return None
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-gptq", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the configs[0] / [2] / [3] blocks and the observer / sparser CPU baselines")
    ap.add_argument("--no-graphs", action="store_true", help="enqueue the 109 launches eagerly instead of replaying CUDA graphs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; --impl reference has none")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch.distributed as dist

    from sparsebit_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback for the product path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()

    # ---- synthetic workload, resident in HBM -------------------------------------------------
    bs = 256
    g = torch.Generator(device=dev).manual_seed(1000 + rank)
    acts, weights = [], []
    for shape, relu in r50_activation_sites(bs):
        x = torch.randn(shape, device=dev, generator=g)
        if relu:
            x.relu_()
        mn, mx = x.min().clamp(max=0), x.max().clamp(min=0)
        s = ((mx - mn) / 255.0).clamp(min=1e-6).reshape(1)
        z = torch.round(-mn / s).reshape(1)
        acts.append((x, torch.empty_like(x), s, z))
    for shape in r50_weight_sites():
        w = torch.randn(shape, device=dev, generator=g) * (2.0 / numel(shape[1:])) ** 0.5
        amax = w.reshape(shape[0], -1).abs().max(dim=1).values
        s = (amax * 2 / 255.0).clamp(min=1e-6).contiguous()
        weights.append((w, torch.empty_like(w), s, torch.zeros_like(s)))
    act_elems = sum(a[0].numel() for a in acts)
    w_elems = sum(w[0].numel() for w in weights)
    assert act_elems == 10_764_800 * bs and w_elems == 25_502_912 and len(acts) == 55 and len(weights) == 54
    step_elems = act_elems + w_elems
    # one contiguous MinMax state array for the 55 observers -> a single init launch per step
    mm_states = torch.empty(2 * len(acts), dtype=torch.int32, device=dev)
    side = torch.cuda.Stream(device=dev)  # CUDA-graph capture needs a non-default stream
    torch.cuda.synchronize()

    def enqueue_acts(stream):
        rc = lib.sb200_minmax_init(mm_states.data_ptr(), len(acts), stream)
        for i, a in enumerate(acts):
            rc |= lib.sb200_qdq_stats_pertensor_fwd(a[0].data_ptr(), a[2].data_ptr(), a[3].data_ptr(), a[1].data_ptr(),
                                                    mm_states.data_ptr() + 8 * i, a[0].numel(), 0, 255, 0, stream)
        if rc:
            _lib.check(rc, "qdq_stats")

    # the 54 weight quantizers of the model run as ONE launch (sb200_qdq_multi_plan once, sb200_qdq_multi_run per step):
    # single layers are L2-resident and launch-bound when issued one by one (54 launches: 0.076 of the HBM roofline)
    from sparsebit_b200 import ops as _sbops

    w_plan = _sbops.QdqMulti([dict(x=w[0], out=w[1], scale=w[2], zero_point=w[3], qmin=-128, qmax=127) for w in weights])

    def enqueue_weights(stream):
        _lib.check(lib.sb200_qdq_multi_run(w_plan.table.data_ptr(), w_plan.count, w_plan.total_rows, stream), "qdq_multi_run")

    # The 109 launches of a step are captured once into two CUDA graphs (activation sites, weight
    # sites) and replayed: the step is a launch-bound inner loop from the host's point of view.
    use_graphs = not args.no_graphs
    captured0 = _lib.launch_count()
    if use_graphs:
        g_act, g_w = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        with torch.cuda.stream(side):
            enqueue_acts(side.cuda_stream)  # eager warm-up on the capture stream
            enqueue_weights(side.cuda_stream)
            side.synchronize()
            with torch.cuda.graph(g_act, stream=side):
                enqueue_acts(torch.cuda.current_stream(dev).cuda_stream)
            with torch.cuda.graph(g_w, stream=side):
                enqueue_weights(torch.cuda.current_stream(dev).cuda_stream)
    # kernels per graph replay = launches issued while capturing (eager warm-up issued the same number)
    kernels_per_step = (_lib.launch_count() - captured0) // 2 if use_graphs else 0
    stream = torch.cuda.current_stream(dev).cuda_stream
    ev_a0 = torch.cuda.Event(enable_timing=True)
    ev_a1 = torch.cuda.Event(enable_timing=True)

    def step(mark=False):
        if mark:
            ev_a0.record()
        if use_graphs:
            g_act.replay()
        else:
            enqueue_acts(stream)
        if mark:
            ev_a1.record()
        if use_graphs:
            g_w.replay()
        else:
            enqueue_weights(stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = _lib.launch_count()
    if os.environ.get("SB200_NCU_RANGE"):
        torch.cuda.profiler.start()  # ncu --profile-from-start off: capture only the timed region
    ev0 = torch.cuda.Event(enable_timing=True)
    ev1 = torch.cuda.Event(enable_timing=True)
    act_ms = 0.0
    ev0.record()
    pending = []
    for _ in range(args.steps):
        step(mark=True)
        # event pairs are read after the loop; re-recording the same pair would lose timings, so
        # collect this step's activation-group time lazily with fresh events every step
        pending.append((ev_a0, ev_a1))
        ev_a0 = torch.cuda.Event(enable_timing=True)
        ev_a1 = torch.cuda.Event(enable_timing=True)
    ev1.record()
    barrier()
    if os.environ.get("SB200_NCU_RANGE"):
        torch.cuda.profiler.stop()
    launches = (_lib.launch_count() - launches0) + kernels_per_step * args.steps
    clocks = sampler.stop() if rank == 0 else None
    total_ms = ev0.elapsed_time(ev1)
    act_ms = sum(a.elapsed_time(b) for a, b in pending)
    tmax = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    total_ms = float(tmax)
    ms_per_step = total_ms / args.steps
    value = world * step_elems / (ms_per_step * 1e-3) / 1e9
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, acts, weights, mm_states)

    # parity spot check of what was just timed (fused kernel's min/max state, on-grid outputs)
    mn, mx = (torch.empty(1, device=dev), torch.empty(1, device=dev))
    lib.sb200_minmax_read(mm_states.data_ptr(), 1, mn.data_ptr(), mx.data_ptr(), stream)
    assert float(mn) == float(acts[0][0].min()) and float(mx) == float(acts[0][0].max()), "fused stats mismatch"

    # ---- roofline of the dominant kernel (fused QDQ + stats), measured inside the timed region --
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    act_launches = 55 * args.steps  # (+1 tiny minmax_init launch per step inside the same event pair)
    alg_bytes_per_launch = act_elems * 8.0 / 55
    avg_launch_s = act_ms * 1e-3 / act_launches
    achieved = alg_bytes_per_launch / avg_launch_s / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                "kernel": "sb200::stream_kernel<MODE_TENSOR,VEC4,DOQ,STORE,STATS> (sb200_qdq_stats_pertensor_fwd)",
                "algorithmic_bytes_per_launch": alg_bytes_per_launch, "avg_launch_us": avg_launch_s * 1e6,
                "kernel_share_of_step": act_ms / (ms_per_step * args.steps), "peak_source": peak_src}
    # DRAM traffic of this kernel: dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed
    # `ncu --set full` capture of this command (profiles/r02_traffic.json, written by scripts/summarize_ncu.py);
    # null when no capture of this round is present.
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))["qdq_stats_pertensor"]
        roofline["traffic"] = float(tr["dram_bytes_per_algorithmic_byte"]) * alg_bytes_per_launch
        roofline["traffic_note"] = tr.get("note")
    except Exception:
        pass
    # headline tensor alone: [256,3,224,224] (308 MB in+out > L2), 30 back-to-back launches
    a0 = (acts[0][0].data_ptr(), acts[0][2].data_ptr(), acts[0][3].data_ptr(), acts[0][1].data_ptr(), mm_states.data_ptr(),
          acts[0][0].numel(), 0, 255, 0, stream)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(5):
        lib.sb200_qdq_stats_pertensor_fwd(*a0)
    e0.record()
    for _ in range(30):
        lib.sb200_qdq_stats_pertensor_fwd(*a0)
    e1.record()
    torch.cuda.synchronize()
    a0_us = e0.elapsed_time(e1) * 1e3 / 30
    a0_gbs = acts[0][0].numel() * 8.0 / (a0_us * 1e-6) / 1e9
    roofline["headline_256x3x224x224"] = {"us": a0_us, "GB/s": a0_gbs, "frac": a0_gbs / peak, "Gelem/s": acts[0][0].numel() / (a0_us * 1e-6) / 1e9}
    # the same tensor through each implementation variant (1 = LDG register pipeline, 2 = TMA ring)
    for variant, name in ((1, "ldg"), (2, "tma")):
        lib.sb200_set_variant(variant)
        for _ in range(5):
            lib.sb200_qdq_stats_pertensor_fwd(*a0)
        e0.record()
        for _ in range(30):
            lib.sb200_qdq_stats_pertensor_fwd(*a0)
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / 30
        roofline["headline_256x3x224x224"][name + "_us"] = us
        roofline["headline_256x3x224x224"][name + "_frac"] = acts[0][0].numel() * 8.0 / (us * 1e-6) / 1e9 / peak
    lib.sb200_set_variant(0)

    # ---- end to end: host buffers through the C-ABI host entry points ---------------------------
    e2e = None
    if not args.no_e2e:
        max_a = max(a[0].numel() for a in acts)
        max_w = max(w[0].numel() for w in weights)
        hx = torch.empty(max_a, dtype=torch.float32).pin_memory()
        hy = torch.empty(max_a, dtype=torch.float32).pin_memory()
        hx.copy_(torch.relu(torch.randn(max_a, generator=torch.Generator().manual_seed(7))))
        hw = torch.randn(max_w).pin_memory()
        hwy = torch.empty(max_w).pin_memory()
        hs = torch.full((2048,), 0.01)
        hz = torch.zeros(2048)
        mm = (ctypes.c_float * 2)()
        a_host = [(hx.data_ptr(), ctypes.c_float(float(a[2])), ctypes.c_float(float(a[3])), hy.data_ptr(), ctypes.addressof(mm),
                   a[0].numel(), 0, 255, 0) for a in acts]
        w_host = [(hw.data_ptr(), hs.data_ptr(), hz.data_ptr(), hwy.data_ptr(), 1, w[0].shape[0], numel(w[0].shape[1:]), -128, 127, 0)
                  for w in weights]

        def e2e_step():
            # asynchronous host-buffer calls: copies of consecutive tensors overlap; one sync per group
            for c in a_host:
                rc = lib.sb200_qdq_pertensor_fwd_host_async(*c)
                if rc:
                    _lib.check(rc, "qdq_host")
            _lib.check(lib.sb200_host_sync(), "host_sync")
            for c in w_host:
                rc = lib.sb200_qdq_perchannel_fwd_host(*c)
                if rc:
                    _lib.check(rc, "qdq_pc_host")

        e2e_steps = max(1, min(args.steps, 3))
        e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step()
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        e2e = {"value": world * step_elems * e2e_steps / float(dt) / 1e9, "unit": UNIT,
               "h2d_bytes_per_step": step_elems * 4 + 2 * 4 * sum(w[0].shape[0] for w in weights),
               "d2h_bytes_per_step": step_elems * 4 + 8 * len(acts), "steps": e2e_steps,
               "numa": numa,
               "api": "sb200_qdq_pertensor_fwd_host_async (+minmax) + sb200_host_sync / sb200_qdq_perchannel_fwd_host, pinned host buffers, H2D+D2H inside"}
        del hx, hy, hw, hwy

    # ---- CPU baseline: the reference's CPU op chain on this box's host cores --------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        elems, times, threads, sample_bs = time_cpu_baseline(reps=5, warmup=1, budget_s=2.0)
        cpu = {"value": elems * len(times) / sum(times) / 1e9, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"all 109 sites at batch {sample_bs} instead of 256 ({elems} elems per pass, {len(times)} passes), torch CPU "
                         "op chain of quant_tensor.py:181-184 + min/max (oracle/torch_port.py)"}

    # ---- secondary metric of BASELINE.json: GPTQ int4 g128 tok/s on the LLaMA-7B linear shapes ----------
    # `reference_cuda_kernel` below is a BASELINE leg like `cpu_baseline`: the reference's own CUDA kernel (built
    # from /root/reference into oracle/_ref/gptq_ref.so by oracle/build_ref.py) timed next to ours, because the
    # north star states this target relative to it (>= 1.0x).  Nothing of ours runs through it.
    gptq = None
    if rank == 0 and world == 1 and not args.no_gptq:
        try:
            sys.path.insert(0, os.path.join(ROOT, "scripts"))
            import bench_gptq

            totals = bench_gptq.run([1, 2048], with_reference=True, quiet=True)
            peaks = json.load(open(peaks_path)) if os.path.exists(peaks_path) else {}
            tf_peak = float(peaks.get("bf16_tflops", 1590.0))
            flops_tok = 2 * 6_476_005_376
            t_pre = totals[(2048, "ours_auto")]
            t_dec = min(totals[(1, "ours_auto")], totals.get((1, "ours_fused_launches"), float("inf")))
            dec_bytes = 6_476_005_376 / 2 + 2 * 4 * 6_476_005_376 / 128  # packed int4 + fp32 scales and zeros (g128)
            gptq = {"config": "LLaMA-7B, all 32 x 7 linears, int4 g128, fp16->fp32 activations, CUDA-graph timed, synthetic packed weights",
                    "decode_tok_s": 1.0 / t_dec, "decode_tok_s_one_launch_per_linear": 1.0 / totals[(1, "ours_auto")],
                    "decode_launches": "q/k/v and gate/up fused into one launch each (sb200_gptq4_matmul_batch_ex): 4 launches per layer, "
                                       "programmatic dependent launch, SB200_GPTQ4_STATIC_WEIGHTS (model weights are constants)",
                    "prefill_2048_tok_s": 2048.0 / t_pre,
                    "prefill_2048_useful_TFLOPs": flops_tok * 2048 / t_pre / 1e12,
                    "roofline_prefill": {"bound": "tensor", "achieved": flops_tok * 2048 / t_pre / 1e12, "peak": tf_peak, "unit": "TFLOP/s",
                                         "frac": flops_tok * 2048 / t_pre / 1e12 / tf_peak,
                                         "kernel": "sb200::gptq4_ts_kernel (tcgen05.mma kind::f16, weight planes in TMEM)",
                                         "note": "useful flops 2*M*K*N; the kernel issues two MMA passes (w_hi and w_lo fp16 planes) to keep "
                                                 "fp32-level accuracy, so the tensor pipe does 2x this work"},
                    "roofline_decode": {"bound": "hbm", "achieved": dec_bytes / t_dec / 1e9, "peak": peak, "unit": "GB/s",
                                        "frac": dec_bytes / t_dec / 1e9 / peak, "algorithmic_bytes_per_token": dec_bytes}}
            try:  # the model path: QuantLinear.forward with fp16 activations (sb200_gptq4_linear_f16_ex), one launch per linear
                f16 = bench_gptq.run_f16_linear(1)
                gptq["decode_f16_linear"] = {"tok_s_one_launch": 1.0 / f16["one_launch"], "tok_s_staged_four_launches": 1.0 / f16["staged"],
                                             "api": "ops.gptq4_linear_f16 (QuantLinear.forward, fp16 in / out incl. bias), one launch per linear"}
            except Exception as e:
                gptq["decode_f16_linear"] = {"error": repr(e)[:160]}
            # end to end through ops.gptq4_matmul with HOST activations: one decoder layer's 7 linears (x from pinned host
            # memory, result read back), scaled to the 32 layers
            try:
                from sparsebit_b200 import ops as _ops

                shapes = [(4096, 4096)] * 4 + [(4096, 11008)] * 2 + [(11008, 4096)]
                gq = torch.Generator(device=dev).manual_seed(5)
                layer = []
                for k_, n_ in shapes:
                    qw = torch.randint(-2**31, 2**31 - 1, (k_ // 8, n_), dtype=torch.int64, device=dev, generator=gq).to(torch.int32)
                    sc = torch.rand(n_, k_ // 128, device=dev, generator=gq) * 0.01 + 0.002
                    layer.append((qw, sc, sc * torch.randint(0, 16, (n_, k_ // 128), device=dev, generator=gq).float()))
                hx = {k_: torch.randn(2048, k_).half().float().pin_memory() for k_ in (4096, 11008)}
                hy = {n_: torch.empty(2048, n_).pin_memory() for n_ in (4096, 11008)}

                def layer_e2e():
                    for (k_, n_), (qw, sc, zr) in zip(shapes, layer):
                        x = hx[k_].to(dev, non_blocking=True)
                        y = torch.zeros(2048, n_, device=dev)
                        _ops.gptq4_matmul(x, qw, y, sc, zr, 128)
                        hy[n_].copy_(y, non_blocking=True)
                    torch.cuda.synchronize()

                layer_e2e()
                t0 = time.perf_counter()
                for _ in range(3):
                    layer_e2e()
                t_layer = (time.perf_counter() - t0) / 3
                gptq["e2e"] = {"prefill_2048_tok_s": 2048.0 / (32 * t_layer), "h2d_bytes_per_layer": sum(2048 * k_ * 4 for k_, _ in shapes),
                               "d2h_bytes_per_layer": sum(2048 * n_ * 4 for _, n_ in shapes),
                               "api": "ops.gptq4_matmul per linear with pinned host activations in / out (7 linears of one layer x 32)"}
                del layer, hx, hy
            except Exception as e:
                gptq["e2e"] = {"error": repr(e)[:160]}
            # CPU baseline: the fp32 unpack + matmul restatement (the reference has no CPU path for this kernel,
            # utils/quant.py:290-296), one 4096 x 4096 linear at M = 1, scaled to all linears
            try:
                import numpy as np

                from oracle import gptq as ogptq

                rng = np.random.default_rng(0)
                qw_h = rng.integers(-2**31, 2**31 - 1, (512, 4096), dtype=np.int64).astype(np.int32)
                sc_h = (rng.random((4096, 32)) * 0.01 + 0.002).astype(np.float32)
                zr_h = (sc_h * rng.integers(0, 16, (4096, 32))).astype(np.float32)
                xh = rng.standard_normal((1, 4096)).astype(np.float32)
                tc, _ = timed_cpu(lambda: ogptq.dequant_matmul(xh, qw_h, np.zeros((1, 4096), np.float32), sc_h, zr_h, 128, dtype=np.float32), 2.0)
                gptq["cpu_baseline"] = {"decode_tok_s": 1.0 / (tc * 6_476_005_376 / (4096 * 4096)), "kind": "port", "cores": 1,
                                        "sample": "oracle.gptq.dequant_matmul (numpy fp32 unpack + matmul), one 4096x4096 g128 linear at M=1, "
                                                  "scaled by the weight count of all 224 linears"}
            except Exception as e:
                gptq["cpu_baseline"] = {"error": repr(e)[:160]}
        except Exception as e:  # the headline line must still be printed
            gptq = {"error": repr(e)[:200]}

    # ---- the other BASELINE configs and the CPU baselines BASELINE.md section 3.1 lists ----------------------------
    extra = {}
    if not args.no_extra:
        def guarded(name, fn):
            try:
                return fn()
            except Exception as e:  # the headline line must still be printed
                return {"error": f"{name}: {e!r}"[:300]}

        extra["calibration_deit"] = guarded("calibration", lambda: block_calibration(dev, world, rank, peak))  # all ranks (collectives)
        if world == 1:
            extra["sparse_4w4a"] = guarded("sparse_4w4a", lambda: block_sparse_4w4a(lib, dev, acts, weights, peak, args.steps))
            del acts, weights
            torch.cuda.empty_cache()
            extra["resnet18_ptq"] = guarded("resnet18_ptq", lambda: block_resnet18_ptq(dev))
            if not args.no_cpu:
                extra["cpu_baselines"] = guarded("cpu_baselines", lambda: block_cpu_baselines(cpu["cores"] if cpu else min(16, host_threads())))

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "global_batch": bs * world, "act_elems_per_gpu": act_elems, "weight_elems_per_gpu": w_elems,
                       "parallelism": f"replicas x{world} (path has no exchange step; no data-path collective)",
                       "l2": "inputs larger than L2: 22 GB working set per step, every site owns its in/out buffers",
                       "launch": "2 CUDA graphs (55 activation launches + 1 state init; the 54 weight sites in ONE multi-tensor launch) replayed per step"
                                 if use_graphs else "eager launches (55 activation launches + 1 init + 1 multi-tensor weight launch)"},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks, "gptq": gptq, **extra,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
