#!/usr/bin/env python
"""bench.py — driver-facing benchmark (contract in the task statement, §④).

    python bench.py --gpus N --steps K --warmup W [--workload msda|...] [--impl reference] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  A "step" is one pass of the hot path over one batch of
synthetic input.  Workloads:

  ape_l_d  (default) BASELINE.json configs[1]: the whole APE-L_D detection forward at 1024², 1203-name
           vocabulary, boxes only, batch 1 per GPU -> images/sec.  Synthetic image, random-init weights
           of the real architecture (380 M parameters), seeded synthetic text features (the text tower
           is a cached input of this path).
  msda     ms_deform_attn forward at the APE-L_D 1024² encoder shape (B=1 per GPU, Q=S=87 296,
           5 levels, 8 heads x 32, 4 points) — BASELINE.json's "ms_deform_attn HBM GB/s"
           half of the metric; algorithmic bytes per call as SURVEY.md §8(d).

`value`   : device-resident inputs, CUDA events on the launching stream, max over ranks.
`e2e`     : same metric through the public operator (torch.ops.ape.ms_deform_attn_forward) with
            HOST (pinned) buffers: H2D of value/loc/attn and D2H of the output inside the timed region.
`roofline`: algorithmic bytes per launch / mean launch duration (CUDA events inside the timed
            region) against MEASURED_PEAKS.json's hbm_gbs (fallback 6650 GB/s, said so).
`cpu_baseline`: the oracle port of the reference's CPU path timed on this box's host cores
            (rank 0, N=1 only).  `--impl reference` runs only that arm.
Multi-GPU: the path shards over images with no data-path collective ("weak" scaling: one image
per GPU); launched by torchrun, NCCL is used only for the barrier and the max-over-ranks reduce.
"""
import argparse
import atexit
import json
import math
import os
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

L5_1024 = [(256, 256), (128, 128), (64, 64), (32, 32), (16, 16)]
H, D, P = 8, 32, 4


def msda_bytes(B, S, Q, L, esize):
    """SURVEY.md §8(d): read value once, loc + attn once, write out once (+ level tables)."""
    return esize * (B * S * H * D + B * Q * H * L * P * 2 + B * Q * H * L * P + B * Q * H * D) + 24 * L


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.index)], stdout=self.f, stderr=subprocess.DEVNULL)
            atexit.register(self._kill)  # an exception before stop() must not leave the sampler running after exit
        except OSError:
            self.p = None

    def _kill(self):
        if self.p is not None and self.p.poll() is None:
            self.p.kill()

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name).read().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1]))
                smax.append(float(r[2]))
            except ValueError:
                continue
            for n, v in zip(names, r[5:9]):
                if v.strip().lower() == "active":
                    reasons.add(n)
        if sm:
            sm.sort()
            out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=max(smax), reasons=sorted(reasons), samples=len(sm))
        return out


DUMP_BUDGET = 60 << 20  # bytes of array data --dump-outputs writes at most: under 64 MB with the .npy headers


def _is_rle(obj):
    return isinstance(obj, list) and obj and all(isinstance(v, dict) and set(v) == {"size", "counts"} for v in obj)


def _leaves(name, obj):
    """(name, host tensor) for every array in a step's result: tensors, Boxes, Instances fields, dict / list / tuple members,
    the bytes of COCO run-length strings and plain numbers.  A list of run-length codes (one per instance) becomes three
    arrays: <name>.counts (every code's bytes, concatenated), <name>.counts_len (bytes per code) and <name>.size ([N, 2])."""
    if _is_rle(obj):
        codes = [c.encode() if isinstance(c, str) else bytes(c) for c in (v["counts"] for v in obj)]
        yield f"{name}.counts", torch.frombuffer(bytearray(b"".join(codes)), dtype=torch.uint8)
        yield f"{name}.counts_len", torch.tensor([len(c) for c in codes], dtype=torch.float64)
        yield f"{name}.size", torch.tensor([list(v["size"]) for v in obj], dtype=torch.float64)
    elif torch.is_tensor(obj):
        yield name, obj.detach().cpu()
    elif hasattr(obj, "get_fields"):
        for k, v in obj.get_fields().items():
            yield from _leaves(f"{name}.{k}", v)
    elif hasattr(obj, "tensor"):
        yield name, obj.tensor.detach().cpu()
    elif isinstance(obj, dict):
        for k, v in obj.items():
            yield from _leaves(f"{name}.{k}", v)
    elif isinstance(obj, (list, tuple)) and obj and all(isinstance(v, (bool, int, float)) for v in obj):
        yield name, torch.tensor(obj, dtype=torch.float64)
    elif isinstance(obj, (list, tuple)):
        for i, v in enumerate(obj):
            yield from _leaves(f"{name}.{i}", v)
    elif isinstance(obj, (bytes, str)):
        yield name, torch.tensor(list(obj.encode() if isinstance(obj, str) else obj), dtype=torch.uint8)
    elif isinstance(obj, (bool, int, float)):
        yield name, torch.tensor(obj, dtype=torch.float64)


def dump_outputs(out, directory):
    """Writes what one step returned to its caller as <directory>/<name>.npy: 16/32-bit floats, booleans and integers of up
    to 16 bits as float32, everything else (float64, wider integers) as float64, so that outputs of two builds compare value
    for value.  When the arrays exceed DUMP_BUDGET, those above 1 MiB are replaced by a seeded sample of flat positions (numpy
    default_rng(0): the same positions for the same shape) that shares the budget left after the small ones; when the small ones
    alone would take more than half of it, every non-empty array is sampled to an equal share."""
    import numpy as np

    os.makedirs(directory, exist_ok=True)
    leaves = [(n.strip(".") or "output", t) for n, t in _leaves("", out)]
    width = [4 if t.element_size() <= 4 and (t.is_floating_point() or t.element_size() <= 2) else 8 for _, t in leaves]
    nbytes = [t.numel() * w for (_, t), w in zip(leaves, width)]
    big = [False] * len(leaves)
    if sum(nbytes) > DUMP_BUDGET:
        big = [b > (1 << 20) for b in nbytes]
        if sum(b for b, g in zip(nbytes, big) if not g) > DUMP_BUDGET // 2:
            big = [b > 0 for b in nbytes]
    share = (DUMP_BUDGET - sum(b for b, g in zip(nbytes, big) if not g)) // max(1, sum(big))
    for (name, t), w, g in zip(leaves, width, big):
        flat = t.reshape(-1)
        if g:
            pos = np.unique(np.random.default_rng(0).integers(0, flat.numel(), share // w))
            flat = flat[torch.from_numpy(pos)]
            print(f"bench: --dump-outputs: {name} {tuple(t.shape)} sampled at {pos.size} positions", file=sys.stderr)
        a = flat.to(torch.float32 if w == 4 else torch.float64).numpy()
        np.save(os.path.join(directory, f"{name}.npy"), a if g else a.reshape(tuple(t.shape)))


def host_threads():
    """Threads for the CPU arms: every core up to 32.  The ops of this path stop scaling around there; with one thread
    per core of a 200-core host the oracle forward measured 136 s per image on the B200 box against 29 s on 8 cores."""
    return max(1, min(os.cpu_count() or 1, 32))


def cpu_reference_arm(steps, warmup):
    """The reference's CPU path for ms_deform_attn = multi_scale_deformable_attn_pytorch
    (ape/layers/multi_scale_deform_attn.py:84-124), as the oracle's port of it (oracle/msda.py:msda_torch), all host threads:
    `warmup` untimed and `steps` timed calls."""
    from oracle import msda as O

    cores = host_threads()
    torch.set_num_threads(cores)
    S = sum(h * w for h, w in L5_1024)
    ins = O.make_inputs(1, S, H, D, L5_1024, P, seed=3)
    value, ss, st, loc, attn = ins
    for _ in range(warmup):
        O.msda_torch(value, ss, loc, attn)
    t0 = time.perf_counter()
    for _ in range(steps):
        out = O.msda_torch(value, ss, loc, attn)
    dt = (time.perf_counter() - t0) / steps
    gbs = msda_bytes(1, S, S, 5, 4) / dt / 1e9
    return {"outputs": out, "value": gbs, "unit": "GB/s", "cores": cores, "kind": "port",
            "sample": f"{steps} full encoder-shape calls after {warmup} warm-up(s) (B=1,Q=S={S},L=5,fp32) of the oracle's port of "
                      "multi_scale_deformable_attn_pytorch, all host threads", "ms_per_step": dt * 1e3}


def fused_msda_bytes(B, S, Q, L, e, eo):
    """Algorithmic bytes of one fused MSDA launch (DESIGN.md): value read once, raw offsets + logits
    read once (instead of materialised locations / weights), fp32 reference points, output written once."""
    return e * B * S * H * D + eo * B * Q * H * L * P * 3 + 4 * B * Q * L * 2 + e * B * Q * H * D + 24 * L


BENCH_SCORE_THRESH = 0.0123  # ~500 of the 1.08 M (query, class) scores of the synthetic-weight model pass (golden image: 500 at 0.012292)


def bench_spec():
    import copy

    from ape_b200 import configs

    spec = copy.deepcopy(configs.APE_L_D)
    spec["test_score_thresh"] = BENCH_SCORE_THRESH
    return spec


def bench_weights(model):
    """Synthetic weights shared by BOTH arms: a pure function of parameter names and shapes (ape_b200/synthetic.py), then the
    proposal-head bias shift that makes invalid anchors score at the prior (as with trained weights)."""
    from ape_b200 import synthetic

    synthetic.fill_state_dict(model)
    synthetic.suppress_invalid_anchor_logits(model)
    return model


def cpu_model_arm(steps, warmup, n_text=1203, sd=None, seed=0):
    """Reference arm for the ape_l_d workload: the oracle's CPU port of the reference forward
    (oracle/ape_forward.py), fp32, up to 32 host threads: `warmup` untimed and `steps` timed forwards.  One whole-image
    forward is ~25 s of host time on the B200 box, so a short run wants a small --steps.  Same spec, same weights, same
    threshold, same image generator as the GPU arm."""
    from ape_b200 import synthetic
    from ape_b200.modeling import build_model
    from oracle import ape_forward as AF

    cores = host_threads()
    torch.set_num_threads(cores)
    spec = bench_spec()
    text = synthetic.text_features(8192, spec["lang_dim"])[:n_text]
    if sd is None:
        m = bench_weights(build_model(spec, num_text=n_text))  # parameter container only; the port is functional over its state_dict
        sd = m.state_dict()
    else:
        sd = {k: v.detach().to("cpu", torch.float32) for k, v in sd.items()}
    img = torch.randint(0, 256, (3, 1024, 1024), generator=torch.Generator().manual_seed(seed)).to(torch.float32)
    for _ in range(warmup):
        AF.forward([img], [(1024, 1024)], text, sd, spec)
    t0 = time.perf_counter()
    for _ in range(steps):
        res, _ = AF.forward([img], [(1024, 1024)], text, sd, spec)
    dt = (time.perf_counter() - t0) / steps
    return {"outputs": res, "value": 1.0 / dt, "unit": "images/s", "cores": cores, "kind": "port",
            "sample": f"{steps} whole-image forward(s) after {warmup} warm-up(s) of the oracle port (APE-L_D 1024^2, {n_text} names, fp32), "
                      f"{cores} threads of {os.cpu_count()} host cores",
            "ms_per_step": dt * 1e3, "detections": int(res[0]["scores"].numel())}



def msda_microbench(dev, quick=False):
    """BASELINE.json config 5 inside the driver-run record: ms_deform_attn forward on 4-level (128^2..16^2) and the
    model's 5-level pyramids, Q in {300, 900, S}, fp32 / fp16 / bf16, L2 flushed before every timed launch, median of 7:
    the drop-in operator (ape_msda_fwd), the engine's fused kernels (generic and pair layout, incl. the pairing pass) and —
    when oracle/_ref/libref_msda.so travelled with the repo — the REFERENCE's own CUDA kernel recompiled for sm_100a on
    identical tensors (measurement only: the 'kernel to beat'; never on the product path)."""
    from ape_b200 import ops

    ref_cuda = None
    try:
        from oracle import msda as O

        if O.have_ref_cuda():
            ref_cuda = O.ref_cuda
    except Exception:  # noqa: BLE001
        ref_cuda = None
    peak, _ = peaks()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def med(fn, iters=7):
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(iters):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        ts.sort()
        return ts[len(ts) // 2]

    L4 = [(128, 128), (64, 64), (32, 32), (16, 16)]
    cases = [("L4_q300", L4, 300), ("L4_q900", L4, 900), ("L4_qS", L4, None), ("L5_1024_q900", L5_1024, 900),
             ("L5_1024_qS", L5_1024, None)]
    if quick:
        cases = [cases[1], cases[4]]
    rows = []
    for name, shapes, Q in cases:
        ss = torch.tensor(shapes, dtype=torch.int64)
        areas = ss[:, 0] * ss[:, 1]
        st = torch.cat([areas.new_zeros(1), areas.cumsum(0)[:-1]])
        S, L = int(areas.sum()), len(shapes)
        q = S if Q is None else Q
        g = torch.Generator().manual_seed(3)
        value = torch.randn(1, S, H, D, generator=g)
        loc = torch.rand(1, q, H, L, P, 2, generator=g)
        logits = torch.randn(1, q, H, L * P, generator=g)
        attn = logits.softmax(-1).view(1, q, H, L, P)
        ssd, std = ss.to(dev), st.to(dev)
        for dname, dt, e in (("f32", torch.float32, 4), ("f16", torch.float16, 2), ("bf16", torch.bfloat16, 2)):
            v, lo, at = (t.to(dev, dt) for t in (value, loc, attn))
            nb = msda_bytes(1, S, q, L, e)
            r = {"case": name, "dtype": dname, "S": S, "Q": q, "L": L, "alg_MB": round(nb / 1e6, 2)}
            t = med(lambda: ops.ms_deform_attn_forward(v, ssd, std, lo, at, 64))
            r["op_ms"], r["op_frac_hbm"] = round(t, 4), round(nb / t / 1e6 / peak, 4)
            if ref_cuda is not None and dt != torch.bfloat16:
                t = med(lambda: ref_cuda(v, ssd, std, lo, at))
                r["reference_kernel_ms"] = round(t, 4)
                r["speedup_vs_reference_kernel"] = round(t / r["op_ms"], 2)
            if dt != torch.float32:
                # engine form: raw offsets (reference point 0, so loc = off / (W,H)) + logits, as the module calls it
                norm = torch.tensor([[w_, h_] for h_, w_ in shapes], dtype=torch.float32)
                offs = (loc * norm[None, None, None, :, None, :]).reshape(1, q, -1)
                qo = torch.cat([offs, logits.reshape(1, q, -1)], -1).to(dev, dt)
                n_off = H * L * P * 2
                ref0 = torch.zeros(1, q, L, 2, device=dev)
                fb = fused_msda_bytes(1, S, q, L, e, e)
                t = med(lambda: ops.ms_deform_attn_fused_forward(v, ssd, std, qo[..., :n_off], qo[..., n_off:], ref0, P))
                r["fused_ms"], r["fused_frac_hbm"] = round(t, 4), round(fb / t / 1e6 / peak, 4)
                if ops.msda_pair_supported(shapes, H, D, P, dt):
                    v3 = v.view(1, S, H * D)
                    t = med(lambda: ops.ms_deform_attn_pair_fused_forward(ops.msda_pair_values(v3, H), ssd, std, shapes,
                                                                          qo[..., :n_off], qo[..., n_off:], ref0, P))
                    r["pair_ms_incl_pairing"], r["pair_frac_hbm"] = round(t, 4), round(fb / t / 1e6 / peak, 4)
                    v2 = ops.msda_pair_values(v3, H)
                    t = med(lambda: ops.ms_deform_attn_pair_fused_forward(v2, ssd, std, shapes, qo[..., :n_off], qo[..., n_off:], ref0, P))
                    r["pair_gather_only_ms"] = round(t, 4)
            rows.append(r)
            del v, lo, at
    return {"peak_GBps": peak, "flush": "256 MiB memset before every timed launch", "reference_kernel": ref_cuda is not None,
            "rows": rows}


def phrase_bench(args, rank, local_rank, world):
    """BASELINE.json configs[3]: APE-L_D at 1536 x 1536, 5 000 free-text phrases ("text" prompt -> "phrase" routing:
    VisionLanguageFusion and the classifier both see N_t = 5 000), batch 4 on one GPU.  Stresses the bi-directional
    fusion attention (S = 196 416 vision tokens x 5 000 phrases x 8 heads of 256: 12 TFLOP per layer and image) and the
    text-feature path.  Reports images/s, the fusion attention's TFLOP/s and the peak device memory."""
    import copy

    assert args.impl != "reference", "the CPU port does not cover the 1536^2 / 5 000-phrase configuration in bounded time"
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback in ape_b200)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    import ape_b200
    from ape_b200 import configs, ops
    from ape_b200.modeling import build_model

    n_phr, B, side = args.phrases, args.batch, 1536
    spec = copy.deepcopy(configs.APE_L_D_1536)
    spec["test_score_thresh"] = BENCH_SCORE_THRESH
    tdt = {"fp32": torch.float32, "fp16": torch.float16, "bf16": torch.bfloat16}[args.dtype]
    model = bench_weights(build_model(spec, num_text=1203)).to(dev)
    model.engine_dtype = tdt
    phrases = ",".join(f"object number {i}" for i in range(n_phr))  # contain spaces -> "phrase" (deformable_detr_segm_vl.py:229-232)
    g = torch.Generator().manual_seed(rank)
    host = [torch.randint(0, 256, (3, side, side), generator=g).to(torch.float32).pin_memory() for _ in range(B)]

    def step(use_host=True):
        imgs = host if use_host else [t.to(dev) for t in host]
        return model([{"image": im, "height": side, "width": side, "prompt": "text", "text_prompt": phrases} for im in imgs])

    torch.cuda.reset_peak_memory_stats()
    for _ in range(max(1, args.warmup)):
        step()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(args.steps):
        out = step()
    b.record()
    torch.cuda.synchronize()
    if args.dump_outputs:
        dump_outputs(out, args.dump_outputs)
    ms = a.elapsed_time(b) / args.steps
    ops.PROFILE_EVENTS = []
    n0 = ape_b200._lib.launch_count()
    step()
    torch.cuda.synchronize()
    launches = ape_b200._lib.launch_count() - n0
    events, ops.PROFILE_EVENTS = ops.PROFILE_EVENTS, None
    own = {}
    for (t, x, y) in events:
        own[t[0]] = own.get(t[0], 0.0) + x.elapsed_time(y)
    xs = [(t, x.elapsed_time(y)) for (t, x, y) in events if t[0] == "attention_cross"]
    # flops of one cross-attention launch: 4 * seqs * heads * nq * n_valid * head_dim (QK^T and PV)
    xflops = sum(4.0 * t[1] * t[4] * t[2] * t[3] * t[5] for t, _ in xs)
    xms = sum(d for _, d in xs)
    clocks = sampler.stop()
    tpeak = 1590.0
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        tpeak = float(json.load(open(pk)).get("bf16_tflops", 0) or 0) or tpeak
    line = {"metric": "images_per_sec", "value": B * 1e3 / ms, "unit": "images/s", "n_gpus": 1, "steps": args.steps,
            "warmup": max(1, args.warmup), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {"fp32": "f32", "fp16": "f16", "bf16": "bf16"}[args.dtype], "data": "synthetic",
            "config": {"workload": f"APE-L_D detection forward, {side}x{side} images, {n_phr} free-text phrases (phrase prompt), batch {B} on one GPU",
                       "weights": "random init of the real architecture", "text": "seeded synthetic phrase features (text tower out of path)"},
            "e2e": {"value": B * 1e3 / ms, "unit": "images/s", "h2d_bytes_per_step": B * 3 * side * side * 4,
                    "d2h_bytes_per_step": int(sum(len(o["instances"]) for o in out) * 36), "ms_per_step": ms,
                    "note": "the timed steps already take pinned host images and return host detections"},
            "roofline": {"bound": "tensor", "achieved": xflops / (xms * 1e-3) / 1e12 if xms > 0 else None, "peak": tpeak, "unit": "TFLOP/s",
                         "frac": (xflops / (xms * 1e-3) / 1e12 / tpeak) if xms > 0 else None, "traffic": None,
                         "kernel": "attn_xfwd_kernel (VisionLanguageFusion, 12 launches per step)", "flops_per_step": xflops, "ms_per_step": xms},
            "gpu_launches": int(launches) * args.steps, "clocks": clocks,
            "peak_memory_GB": torch.cuda.max_memory_allocated() / 2 ** 30,
            "own_kernel_ms_per_step": {k: round(v, 2) for k, v in sorted(own.items(), key=lambda kv: -kv[1])},
            "detections": [len(o["instances"]) for o in out]}
    print(json.dumps(line))


def model_bench(args, rank, local_rank, world):
    n_text = 1203
    # identical in both arms (the driver compares it): nothing below depends on which implementation runs
    config = {"workload": "APE-L_D detection forward, 1024x1024 image, 1203-name vocabulary, boxes only, batch 1 per GPU",
              "weights": "random init of the real architecture (380 M params): ape_b200/synthetic.py, invalid anchors at the 0.01 prior",
              "text": "seeded synthetic features (text tower out of path)",
              "l2": "per-step working set (weights 0.75 GB 16-bit + activations) >> 126 MB L2",
              "selection": f"test_score_thresh {BENCH_SCORE_THRESH} (~500 of 1.08M scores pass with these weights; README recipe: 0.1 "
                           "with trained weights); NMS 0.7; top-300",
              "parallelism": f"dp{args.gpus} (one image per GPU; one NCCL gather of packed detections per step when N>1)"}
    if args.impl == "reference":
        if rank != 0:
            return
        os.environ["APE_B200_CONTAINER_ONLY"] = "1"  # parameter containers only: libape_b200.so is not mapped in this arm
        cb = cpu_model_arm(args.steps, args.warmup, n_text)
        if args.dump_outputs:
            dump_outputs(cb["outputs"], args.dump_outputs)
        print(json.dumps({"impl": "reference", "metric": "images_per_sec", "value": cb["value"], "unit": "images/s",
                          "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                          "ms_per_step": cb["ms_per_step"],
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                          "data": "synthetic", "config": config, "detections_per_image": cb["detections"],
                          "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
                          "e2e": {"value": cb["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback in ape_b200)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    import ape_b200
    from ape_b200 import ops
    from ape_b200.modeling import build_model

    from ape_b200 import synthetic

    tdt = {"fp32": torch.float32, "fp16": torch.float16, "bf16": torch.bfloat16}[args.dtype]
    model = bench_weights(build_model(bench_spec(), num_text=n_text)).to(dev)
    model.engine_dtype = tdt  # parameters stay fp32; 16-bit = tensor-core engine path
    model.use_cuda_graphs = tdt != torch.float32 and not args.no_graphs
    masks_on = args.workload == "ape_l_d_masks"  # BASELINE.json configs[2]: boxes + instance masks + semantic map
    if masks_on:
        model.test_mask_on, model.semantic_on = True, True
        model.mask_format = args.mask_format  # "rle": the pasted masks leave as COCO run-length codes (what the evaluators encode them into)
        if args.mask_format == "rle":
            config["mask_format"] = "COCO run-length codes computed on the device (pred_masks_rle) instead of [N,H,W] booleans"
        config["workload"] = config["workload"].replace("boxes only", "boxes + instance masks (128^2 per box, pasted) + semantic map (1203 x 1024^2)")
    g = torch.Generator().manual_seed(rank)
    NIMG = 4
    host_imgs = [torch.randint(0, 256, (3, 1024, 1024), generator=g).to(torch.float32).pin_memory() for _ in range(NIMG)]
    dev_imgs = [t.to(dev) for t in host_imgs]

    from ape_b200 import parallel

    def step(i, host):
        img = host_imgs[i % NIMG] if host else dev_imgs[i % NIMG]
        inputs = [{"image": img, "height": 1024, "width": 1024}]
        if world > 1 and masks_on:  # masks stay on their rank (evaluators consume them there); boxes go to rank 0
            out = model(inputs)
            parallel.gather_detections([o["instances"] for o in out], 300, dev, dst=0)
            return out
        if world > 1:
            # the one collective of the path: the packed detections stay on the device and go straight into ONE NCCL gather
            # on the compute stream; only rank 0 copies to the host (no per-rank D2H / Python packing / H2D round trip)
            out = parallel.gather_packed(model.forward_packed(inputs), dst=0)
            if out is None:
                torch.cuda.current_stream().synchronize()  # a step ends when this rank's contribution has left
            return out
        return model(inputs)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    warm = max(args.warmup, 3)
    for i in range(warm):
        step(i, False)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    a.record()
    for i in range(args.steps):
        out = step(i, False)
    b.record()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(out, args.dump_outputs)
    total_ms = a.elapsed_time(b)
    # Per-kernel durations for the roofline object: CUDA events cannot be recorded inside a graph replay, so
    # the same steps are run a few more times eagerly (same kernels, same inputs, same stream) with an event
    # pair around every launch of our library; launches per step are counted here too.
    def local(i):  # the rank's own forward without the collective (per-kernel / per-stage profiling passes)
        return model([{"image": dev_imgs[i % NIMG], "height": 1024, "width": 1024}])

    model.profile_stages = True
    stage_acc = {}
    for i in range(5):
        local(i)
        for k, v in model.stage_ms.items():
            stage_acc[k] = stage_acc.get(k, 0.0) + v / 5
    model.profile_stages = False
    graphs_on, model.use_cuda_graphs = model.use_cuda_graphs, False
    local(0)
    barrier()
    ops.PROFILE_EVENTS = []
    n0 = ape_b200._lib.launch_count()
    prof_steps = 3
    for i in range(prof_steps):
        # keep the GPU busy while the host enqueues the (un-graphed) step, so every event pair brackets device time only
        # and not the host's launch latency (a 10 us kernel otherwise reads ~18 us when the GPU is waiting for the host)
        try:
            torch.cuda._sleep(int(1.2e8))
        except Exception:  # noqa: BLE001  (private helper; the numbers are then upper bounds for short kernels)
            pass
        local(i)
    barrier()
    launches = (ape_b200._lib.launch_count() - n0) // prof_steps * args.steps
    events, ops.PROFILE_EVENTS = ops.PROFILE_EVENTS, None
    model.use_cuda_graphs = graphs_on
    engine = {"cuda_graphs": bool(graphs_on), "engine_dtype": args.dtype,
              "residual_stream": "fp32 (GEMM epilogues write fp32 sums; operands and LayerNorm outputs 16-bit)"}
    own_ms = {}
    for (t, x, y) in events:
        own_ms[t[0]] = own_ms.get(t[0], 0.0) + x.elapsed_time(y) / prof_steps
    own_ms = {k: round(v, 3) for k, v in sorted(own_ms.items(), key=lambda kv: -kv[1])}
    # tensor-core side of the step: all GEMM launches (2*M*N*K flops each) and the ViT attention launches
    # (4*seq*heads*n*n*64 flops) against the measured cuBLAS bf16 peak of this pool
    # GEMMs with at least 2048 rows: their device time dwarfs the host's launch gap, which an event pair in this eager pass cannot
    # separate from a 7 us kernel (the 900-row decoder GEMMs: latency-bound, < 3 % of the step's GEMM flops, left out and said so)
    gemm_flops_all = sum(2.0 * t[1] * t[2] * t[3] for (t, x, y) in events if t[0] == "gemm_tn") / prof_steps
    gemm_flops = sum(2.0 * t[1] * t[2] * t[3] for (t, x, y) in events if t[0] == "gemm_tn" and t[1] >= 2048) / prof_steps
    gemm_ms = sum(x.elapsed_time(y) for (t, x, y) in events if t[0] == "gemm_tn" and t[1] >= 2048) / prof_steps
    attn_flops = sum(4.0 * t[1] * t[3] * t[2] * t[2] * 64 for (t, x, y) in events if t[0] == "attention") / prof_steps
    attn_ms = sum(x.elapsed_time(y) for (t, x, y) in events if t[0] == "attention") / prof_steps
    enc = [(t, x.elapsed_time(y)) for (t, x, y) in events if t[0] == "msda_fused" and t[3] == t[2]]
    pairing_ms = sum(x.elapsed_time(y) for (t, x, y) in events if t[0] == "msda_pair_values") / max(1, len(enc))
    dec = [(t, x.elapsed_time(y)) for (t, x, y) in events if t[0] == "msda_fused" and t[3] != t[2]]
    # e2e: pinned host image in, detections out on the host (the model's public call does both)
    e2e_steps = max(3, min(args.steps, 10))
    step(0, True)
    barrier()
    a.record()
    for i in range(e2e_steps):
        out = step(i, True)
    b.record()
    barrier()
    e2e_ms = a.elapsed_time(b) / e2e_steps
    # the same image through the predictor (ape_b200.engine.DefaultPredictor, the reference's demo entry): uint8 HWC BGR in,
    # resize on the device (bit-exact with PIL), detections out on the host
    pred_ms, pred_h2d = None, None
    if world == 1:
        import numpy as np

        from ape_b200.engine import DefaultPredictor, ResizeShortestEdge

        predictor = DefaultPredictor(model, ResizeShortestEdge(1024, 1024), "RGB")
        u8 = [np.random.default_rng(100 + i).integers(0, 256, (1024, 1024, 3), dtype=np.uint8) for i in range(NIMG)]
        predictor(u8[0])
        barrier()
        a.record()
        for i in range(e2e_steps):
            predictor(u8[i % NIMG])
        b.record()
        barrier()
        pred_ms, pred_h2d = a.elapsed_time(b) / e2e_steps, int(u8[0].size)
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([total_ms, e2e_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, e2e_ms = t.tolist()
    if rank == 0:
        ms_per_step = total_ms / args.steps
        peak, peak_src = peaks()
        tag, _ = enc[0]
        _, B, S, Q, L, _, e, eo = tag
        enc_ms = sum(x for _, x in enc) / len(enc) + pairing_ms  # one logical op = pairing pass + gather kernel
        nbytes = fused_msda_bytes(B, S, Q, L, e, eo)
        achieved = nbytes / (enc_ms * 1e-3) / 1e9
        lsu_bytes = B * Q * H * L * P * 4 * D * e
        props = torch.cuda.get_device_properties(dev)
        lsu_peak = props.multi_processor_count * 128 * float((clocks or {}).get("sm_max_mhz") or 1965.0) * 1e6 / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get(f"msda_fused_enc_{args.dtype}")
        inst = out[0]["instances"]
        def field_bytes(v):
            if hasattr(v, "tensor"):
                return v.tensor.numel() * 4
            if isinstance(v, list):  # run-length codes: the boundary positions crossed as int32, 4 bytes per run
                return sum(4 * len(r["counts"]) for r in v)
            return v.numel() * v.element_size()

        d2h = sum(field_bytes(v) for v in inst.get_fields().values()) if world == 1 else world * 300 * 13 * 4
        line = {
            "metric": "images_per_sec", "value": world * 1e3 / ms_per_step, "unit": "images/s", "n_gpus": world,
            "steps": args.steps, "warmup": warm, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": {"fp32": "f32", "fp16": "f16", "bf16": "bf16"}[args.dtype], "data": "synthetic",
            "config": config, "engine": engine,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src, "kernel": "msda_pair_fused_kernel + msda_pair_values_kernel (encoder, Q=S)" if pairing_ms > 0
                         else "msda_fused_fwd_kernel (encoder, Q=S)", "pairing_pass_ms": pairing_ms,
                         "algorithmic_bytes_per_launch": nbytes, "launch_ms": enc_ms,
                         "launches_per_step": len(enc) / prof_steps,
                         "share_of_step": enc_ms * len(enc) / prof_steps / ms_per_step,
                         "timing": "event pairs around each launch in 3 eager (non-graph) repeats of the step",
                         "decoder_launch_ms": (sum(x for _, x in dec) / len(dec)) if dec else None,
                         # the bound this gather actually works against: every sample moves 4 corner rows (2 paired 128-byte
                         # lines) through the L1 / LSU data pipe, 128 B/clk/SM (DESIGN.md 5.1.1)
                         "lsu_bytes_per_launch": lsu_bytes, "lsu_peak_GBps": lsu_peak,
                         "lsu_frac": lsu_bytes / (enc_ms * 1e-3) / 1e9 / lsu_peak},
            "e2e": {"value": world * 1e3 / e2e_ms, "unit": "images/s", "h2d_bytes_per_step": host_imgs[0].numel() * 4,
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_ms},
            "e2e_predictor": None if pred_ms is None else {"value": 1e3 / pred_ms, "unit": "images/s", "ms_per_step": pred_ms,
                                                           "h2d_bytes_per_step": pred_h2d, "call": "DefaultPredictor(bgr uint8 HWC image)"},
            "gpu_launches": int(launches), "clocks": clocks,
            "stage_ms_eager_profile": {k: round(v, 3) for k, v in stage_acc.items()},  # un-graphed profiling pass, not the timed path
            "own_kernel_ms_per_step": own_ms,
        }
        tpeak = None
        pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(pk):
            tpeak = float(json.load(open(pk)).get("bf16_tflops", 0) or 0) or None
        tpeak_src = "measured (MEASURED_PEAKS.json bf16_tflops, burst)" if tpeak else "fallback (B200_PROFILING.md 1590 TFLOP/s)"
        tpeak = tpeak or 1590.0
        if gemm_ms > 0:
            a = gemm_flops / (gemm_ms * 1e-3) / 1e12
            line["roofline_gemm"] = {"bound": "tensor", "achieved": a, "peak": tpeak, "unit": "TFLOP/s", "frac": a / tpeak,
                                     "peak_source": tpeak_src,
                                     "kernel": "gemm_tc_kernel / gemm_pair_kernel (every linear layer with >= 2048 rows: "
                                               f"{100.0 * gemm_flops / max(gemm_flops_all, 1.0):.1f} % of the step's GEMM flops)",
                                     "flops_per_step": gemm_flops, "ms_per_step": gemm_ms,
                                     "timing": "event pairs around each launch in eager repeats of the step, enqueued behind a GPU-side delay so the pairs see device time only"}
        if attn_ms > 0:
            a = attn_flops / (attn_ms * 1e-3) / 1e12
            line["roofline_attention"] = {"bound": "tensor", "achieved": a, "peak": tpeak, "unit": "TFLOP/s", "frac": a / tpeak,
                                          "peak_source": tpeak_src, "kernel": "attn_fwd_kernel (24 ViT blocks)",
                                          "flops_per_step": attn_flops, "ms_per_step": attn_ms}
        if world == 1 and not args.no_microbench:
            line["msda_microbench"] = msda_microbench(dev, quick=args.quick_microbench)
        if world == 1 and not args.no_cpu_baseline:
            cb = cpu_model_arm(1, 0, n_text, sd=model.state_dict(), seed=rank)
            line["detections_per_image"] = {"engine": len(inst), "cpu_port": cb["detections"]}
            line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default="ape_l_d", choices=["ape_l_d", "ape_l_d_masks", "msda", "ape_l_d_1536_phrase"])
    ap.add_argument("--phrases", type=int, default=5000, help="ape_l_d_1536_phrase: number of free-text phrases")
    ap.add_argument("--batch", type=int, default=4, help="ape_l_d_1536_phrase: images per step")
    ap.add_argument("--impl", default="ape_b200", choices=["ape_b200", "reference"])
    ap.add_argument("--dtype", default="fp16", choices=["fp32", "fp16", "bf16"])
    ap.add_argument("--mask-format", default="bitmask", choices=["bitmask", "rle"], help="ape_l_d_masks: instance masks as booleans (reference contract) or COCO RLE")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-microbench", action="store_true", help="skip the config-5 ms_deform_attn microbench keys")
    ap.add_argument("--quick-microbench", action="store_true")
    ap.add_argument("--no-graphs", action="store_true", help="disable CUDA-graph capture of the static stages")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 0:
        ap.error("--warmup must be at least 0")
    if args.dump_outputs and os.path.isdir(args.dump_outputs) and os.listdir(args.dump_outputs):
        ap.error(f"--dump-outputs: {args.dump_outputs} is not empty (files of an earlier dump would mix with this one)")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    S = sum(h * w for h, w in L5_1024)
    L = len(L5_1024)
    tdt = {"fp32": torch.float32, "fp16": torch.float16, "bf16": torch.bfloat16}[args.dtype]
    esize = 4 if args.dtype == "fp32" else 2
    config = {"workload": "ms_deform_attn_forward APE-L_D 1024^2 encoder shape (B=1/GPU, Q=S=87296, L=5, H=8, D=32, P=4)",
              "loc": "uniform(0,1) seed 3 (SURVEY 8d)", "l2": "4 rotating input sets (1.4 GB fp32) > 126 MB L2",
              "parallelism": f"dp{args.gpus} (one image per GPU, no data-path collective)"}

    if args.workload in ("ape_l_d", "ape_l_d_masks"):
        return model_bench(args, rank, local_rank, world)
    if args.workload == "ape_l_d_1536_phrase":
        return phrase_bench(args, rank, local_rank, world)

    if args.impl == "reference":
        if rank != 0:
            return
        cb = cpu_reference_arm(args.steps, args.warmup)
        if args.dump_outputs:
            dump_outputs(cb["outputs"], args.dump_outputs)
        line = {"impl": "reference", "metric": "ms_deform_attn_algorithmic_GBps", "value": cb["value"], "unit": "GB/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_step"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config,
                "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": cb["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback in ape_b200)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    import ape_b200
    from ape_b200 import ops

    # --- inputs: 4 rotating sets so consecutive steps never hit a warm L2 -------------------
    NSETS = 4
    g = torch.Generator().manual_seed(3 + rank)
    ss = torch.tensor(L5_1024, dtype=torch.int64)
    areas = ss[:, 0] * ss[:, 1]
    st = torch.cat([areas.new_zeros(1), areas.cumsum(0)[:-1]])
    ss_d, st_d = ss.to(dev), st.to(dev)
    host_sets, dev_sets = [], []
    for i in range(NSETS):
        value = torch.randn(1, S, H, D, generator=g).to(tdt)
        loc = torch.rand(1, S, H, L, P, 2, generator=g).to(tdt)
        attn = torch.randn(1, S, H, L * P, generator=g).softmax(-1).view(1, S, H, L, P).to(tdt)
        host_sets.append(tuple(t.pin_memory() for t in (value, loc, attn)))
        dev_sets.append(tuple(t.to(dev) for t in (value, loc, attn)))

    def step(i):
        v, lo, at = dev_sets[i % NSETS]
        return ops.ms_deform_attn_forward(v, ss_d, st_d, lo, at, 64)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for i in range(max(args.warmup, 3)):
        step(i)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    n0 = ape_b200._lib.launch_count()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_start.record()
    for i in range(args.steps):
        evs[i][0].record()
        out = step(i)
        evs[i][1].record()
    t_end.record()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(out, args.dump_outputs)
    launches = ape_b200._lib.launch_count() - n0
    total_ms = t_start.elapsed_time(t_end)
    kern_ms = sum(a.elapsed_time(b) for a, b in evs) / args.steps

    # --- e2e: host buffers in, host result out, through the public operator ----------------
    out_host = torch.empty((1, S, H * D), dtype=tdt).pin_memory()
    e2e_steps = max(3, min(args.steps, 10))

    def e2e_step(i):
        hv, hl, ha = host_sets[i % NSETS]
        v = hv.to(dev, non_blocking=True)
        lo = hl.to(dev, non_blocking=True)
        at = ha.to(dev, non_blocking=True)
        out = torch.ops.ape.ms_deform_attn_forward(v, ss_d, st_d, lo, at, 64)
        out_host.copy_(out, non_blocking=True)

    e2e_step(0)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(e2e_steps):
        e2e_step(i)
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1) / e2e_steps
    clocks = sampler.stop() if rank == 0 else None

    # max over ranks
    t = torch.tensor([total_ms, kern_ms, e2e_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, kern_ms, e2e_ms = t.tolist()

    if rank == 0:
        nbytes = msda_bytes(1, S, S, L, esize)
        ms_per_step = total_ms / args.steps
        value_gbs = world * nbytes / (ms_per_step * 1e-3) / 1e9
        peak, peak_src = peaks()
        achieved = nbytes / (kern_ms * 1e-3) / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get(f"msda_enc_{args.dtype}")
        h2d = sum(t.numel() * t.element_size() for t in host_sets[0])
        d2h = out_host.numel() * out_host.element_size()
        line = {
            "metric": "ms_deform_attn_algorithmic_GBps", "value": value_gbs, "unit": "GB/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": {"fp32": "f32", "fp16": "f16", "bf16": "bf16"}[args.dtype],
            "data": "synthetic", "config": config,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src, "kernel": "msda_fwd_kernel",
                         "algorithmic_bytes_per_launch": nbytes, "launch_ms": kern_ms},
            "e2e": {"value": world * nbytes / (e2e_ms * 1e-3) / 1e9, "unit": "GB/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms},
            "gpu_launches": int(launches), "clocks": clocks,
        }
        if world == 1 and not args.no_cpu_baseline:
            cb = cpu_reference_arm(2, 1)
            line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
